"""Parity of the BENCHED workload itself (SURVEY §8d config 2: "first 1M lanes replayed through the oracle"): the exact
1,048,576-lane U{0..20}-ply connect_four batch bench.py times (same builder, same seed) is replayed lane by lane on the
UNMODIFIED reference, and every output of the benched step — legal mask before, terminal, current player, returns, next
legal mask and the full observation tensor after — must match on every lane.  The reference's outputs are stored as
digests (tests/reference_golden.py), with digests of the batch they were computed on.  Both host entry points (float and
compact) are checked on the same batch."""
import os
import sys

import numpy as np
import pytest
import torch

from reference_golden import digest, expected

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pytestmark = pytest.mark.gpu


def benched_batch():
    import bench
    import open_spiel_b200 as b2
    game = b2.Game("connect_four", device=0)
    _, snap, actions, hist = bench.build_workload(torch, game, bench.N_STATES, torch.device("cuda", 0), seed=0x5EED,
                                                  with_history=True)
    return game, snap, actions, hist


def reference_golden():
    """Needs a CUDA device: the batch is built there, as bench.py builds it, and replayed on the reference."""
    import ref_lib
    _, _, actions, hist = benched_batch()
    hist, actions = hist.cpu().numpy(), actions.cpu().numpy()
    ref = ref_lib.replay_batch("connect_four", hist, actions, mask_words=1)
    assert ref["failed_lanes"] == 0
    out = {"batch": digest(hist, actions), "terminal_count": int(ref["terminal"].sum())}
    out.update({k: digest(ref[k]) for k in ("mask_before", "terminal", "cur_player", "returns", "mask_after", "obs_bits")})
    return {"gpu_bench_workload/connect_four": out}


def test_benched_connect_four_batch_equals_reference_on_every_lane():
    import bench
    ref = expected("gpu_bench_workload/connect_four")
    n = bench.N_STATES
    dev = torch.device("cuda", 0)
    game, snap, actions, hist = benched_batch()
    assert hist.shape == (n, bench.MAX_PREFIX)
    assert digest(hist.cpu().numpy(), actions.cpu().numpy()) == ref["batch"]      # the batch the reference replayed
    # the device step on the benched batch
    work = game.new_batch(n)
    work.copy_from(snap)
    mask_before = work.legal_actions_mask_words().cpu().numpy().astype(np.uint32)
    mask = torch.empty((n, 1), dtype=torch.int32, device=dev)
    term = torch.empty((n,), dtype=torch.uint8, device=dev)
    rets = torch.empty((n, 2), dtype=torch.float32, device=dev)
    work.step(actions, mask, term, rets)
    work.check_errors()
    cur, term2, rets2 = work.status()
    obs = work.observation_tensor(player=0)                       # [n, 126] float32
    assert digest(mask_before) == ref["mask_before"]
    terminal = term.cpu().numpy()
    assert digest(terminal) == ref["terminal"] and np.array_equal(term2.cpu().numpy(), terminal)
    assert digest(cur.cpu().numpy()) == ref["cur_player"]
    returns = rets.cpu().numpy()
    assert digest(returns) == ref["returns"] and np.array_equal(rets2.cpu().numpy(), returns)
    mask_after = mask.cpu().numpy().astype(np.uint32)
    assert digest(mask_after) == ref["mask_after"]
    F = obs.shape[1]
    pad = torch.zeros((n, (-F) % 32), dtype=obs.dtype, device=dev)
    bits = (torch.cat([obs, pad], dim=1) != 0).reshape(n, -1, 32).to(torch.int64)
    words = (bits << torch.arange(32, device=dev, dtype=torch.int64)).sum(dim=2).cpu().numpy().astype(np.uint32)
    assert digest(words) == ref["obs_bits"]
    assert ref["terminal_count"] == int(terminal.sum()) > 0 and int((terminal == 0).sum()) > n // 2   # the step does end some games
    # the two host entry points on the same batch, against the outputs just matched with the reference
    work.copy_from(snap)
    act_h = actions.cpu().pin_memory()
    mask_h = torch.empty((n, 1), dtype=torch.int32).pin_memory()
    term_h = torch.empty((n,), dtype=torch.uint8).pin_memory()
    rets_h = torch.empty((n, 2), dtype=torch.float32).pin_memory()
    torch.cuda.synchronize()
    work.step_host(act_h, mask_h, term_h, rets_h)
    assert np.array_equal(term_h.numpy(), terminal) and np.array_equal(rets_h.numpy(), returns)
    assert np.array_equal(mask_h.numpy().astype(np.uint32), mask_after)
    work.copy_from(snap)
    torch.cuda.synchronize()
    status_h = torch.empty((n,), dtype=torch.uint8).pin_memory()
    work.step_host_compact(actions.to(torch.uint8).cpu().pin_memory(), status_h)
    st = status_h.numpy()
    t = terminal.astype(bool)
    assert np.array_equal(st >> 7, terminal)
    assert np.array_equal(st[~t] & 0x7F, mask_after[~t, 0].astype(np.uint8))
    outcome = np.where(returns[:, 0] > 0, 1, np.where(returns[:, 0] < 0, 2, 0)).astype(np.uint8)
    assert np.array_equal(st[t] & 3, outcome[t])
    work.check_errors()


@pytest.mark.parametrize("n", [1, 3, 5, 33])
@pytest.mark.parametrize("gs", ["tic_tac_toe", "kuhn_poker", "leduc_poker", "connect_four", "hex(board_size=3)"])
def test_observation_rows_need_no_16_byte_alignment(gs, n):
    """ADVICE r01 (high): k_obs emits float4 stores; row t of the trajectory recorder starts at t*n*F floats, which is
    16-byte aligned only when n*F % 4 == 0.  Odd batch sizes must work and agree with the aligned call."""
    import open_spiel_b200 as b2
    game = b2.load_game(gs)
    batch = game.new_batch(n)
    tr = batch.record_trajectories(seed=5)
    assert batch.error_count()[0] == 0
    obs = tr.time_major["observations"]                      # [T, n, F]
    batch2 = game.new_batch(n)
    tr2 = batch2.record_trajectories(seed=5, include_full_observations=False)
    assert torch.equal(tr.time_major["actions"], tr2.time_major["actions"])
    # the first row is the tensor of the start state (after the initial chance moves): recompute it with an aligned buffer
    b3 = game.new_batch(n)
    F = obs.shape[2]
    base = torch.zeros((n * F + 8,), dtype=torch.float32, device=obs.device)
    for shift in (0, 1, 2, 3):                                # every 4-byte phase of the output pointer
        out = base[shift:shift + n * F].view(n, F)
        which = b3.information_state_tensor if b3.info.information_state_tensor_size > 0 else b3.observation_tensor
        if b3.info.max_chance_outcomes == 0:
            which(player=-1, out=out)
            assert torch.equal(out, obs[0]), (gs, n, shift)
    torch.cuda.synchronize()

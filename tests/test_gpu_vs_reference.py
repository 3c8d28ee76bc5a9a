"""GPU parity directly against the UNMODIFIED reference: the same lock-step harness as test_gpu_parity_games.py with the
real open_spiel::State objects as the checker, their side stored as a digest (tests/reference_golden.py).
Also: size-independent properties at full batch sizes, and ragged / empty batches."""
import numpy as np
import pytest
import torch

import open_spiel_b200 as b2
from parity import checker_digest, lockstep
from reference_golden import expected

pytestmark = pytest.mark.gpu

GAMES = [("tic_tac_toe", 128), ("connect_four", 128), ("breakthrough", 64), ("hex", 32), ("hex(board_size=4,swap=True)", 64),
         ("go(board_size=9)", 32), ("go(board_size=5)", 64), ("kuhn_poker", 128), ("leduc_poker", 256),
         ("mnk", 16), ("mnk(m=5,n=4,k=3)", 64), ("othello", 64), ("y(board_size=9)", 64), ("havannah(board_size=4,swap=True)", 64), ("havannah", 16)]


def reference_golden():
    import ref_lib
    return {"gpu_vs_reference/" + gs: checker_digest(gs, ref_lib.RefGame, n_lanes=lanes, seed=99,
                                                     check_info_state=gs in ("kuhn_poker", "leduc_poker")) for gs, lanes in GAMES}


@pytest.mark.parametrize("gs,lanes", GAMES, ids=[g for g, _ in GAMES])
def test_device_equals_unmodified_reference(gs, lanes):
    steps, digest = lockstep(gs, n_lanes=lanes, seed=99, checker=None, check_info_state=gs in ("kuhn_poker", "leduc_poker"))
    assert digest == expected("gpu_vs_reference/" + gs)
    assert steps > lanes


@pytest.mark.parametrize("gs,n", [("go(board_size=9)", 1 << 17), ("hex", 1 << 18), ("breakthrough", 1 << 20),
                                  ("tic_tac_toe", 1 << 20), ("leduc_poker", 1 << 20), ("kuhn_poker", 1 << 20),
                                  ("mnk", 1 << 17), ("othello", 1 << 18)])
def test_full_size_rollout_properties(gs, n):
    game = b2.load_game(gs)
    b = game.new_batch(n)
    rets, plies = b.rollout(seed=123)
    cur, term, rets2 = b.status()
    assert bool(term.all()) and bool((cur == -4).all())
    assert torch.equal(rets, rets2)
    assert bool((rets.sum(dim=1) == 0).all())                                   # all seven games are zero-sum
    assert int(plies.max()) <= game.max_game_length() + (3 if "poker" in gs else 0)   # + chance deals
    assert float(rets.abs().max()) <= game.max_utility()
    assert int(b.legal_actions_mask_words().abs().sum()) == 0                   # LegalActions() empty at terminal
    if gs == "hex":
        assert bool((rets[:, 0].abs() == 1).all())                             # no draws in hex
    if gs.startswith("go"):
        assert int(plies.min()) >= 2                                            # IsTerminal needs two moves (go.cc:226)
    # determinism + lane_offset sharding: the second half replayed on its own matches
    half = n // 2
    b2_ = game.new_batch(half)
    r3, p3 = b2_.rollout(seed=123, lane_offset=half)
    assert torch.equal(r3, rets[half:]) and torch.equal(p3, plies[half:])


def test_ragged_and_empty_batches():
    game = b2.load_game("connect_four")
    b = game.new_batch(1000)
    acts = torch.full((1000,), 3, dtype=torch.int32, device=b._dev)
    b.apply_actions(acts, n=0)                                   # n = 0: nothing happens
    b.apply_actions(acts, n=17)                                  # only the first 17 lanes move
    cur, _, _ = b.status()
    assert cur[:17].tolist() == [1] * 17 and cur[17:].tolist() == [0] * 983
    m = b.legal_actions_mask_words(n=5)
    assert m.shape == (5, 1)
    obs = b.observation_tensor(0, n=33)                          # a ragged last warp tile (33 = 32 + 1)
    assert obs.shape == (33, 126) and float(obs[16].sum()) == 42 and float(obs[32].sum()) == 42
    assert float(obs[0, 3]) == 1.0 and float(obs[20, 3]) == 0.0
    with pytest.raises(b2.SpielError):
        b.apply_actions(acts, n=1001)                            # beyond capacity
    b.reset(n=10)                                                # partial reset
    cur, _, _ = b.status()
    assert cur[:10].tolist() == [0] * 10 and cur[10:17].tolist() == [1] * 7

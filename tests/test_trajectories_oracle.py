"""CPU: pins the oracle's trajectory recorder (oracle/algorithms/trajectories.cc) to the UNMODIFIED reference's
RecordBatchedTrajectory (algorithms/trajectories.cc:98-200, built by oracle/ref_build.mk).  The two draw from different
random streams, so every reference episode is lined up by replaying its own action sequence through the oracle
recorder (forced mode): the chance outcomes, which the reference does not record, are read off the information-state
tensors (private card one-hots of both players, public card one-hot in leduc's second round).  All recorded fields
and the padding convention must then agree exactly.  The reference's batch is stored (tests/reference_golden.py): the action
sequences read off each episode, and a digest of every recorded field."""
import numpy as np
import pytest

from oracle_lib import OracleGame, oracle_record_trajectory
from reference_golden import Digest, expected

FIELDS = ("legal_actions", "observations", "actions", "player_ids", "valid", "next_is_terminal", "rewards", "player_policies")
B = 300


def _kuhn_sequence(ep):
    # infostate tensor (kuhn_poker.cc:72-107): player one-hot(2) . card one-hot(3) . betting
    card = {}
    for t in range(len(ep["valid"])):
        if ep["valid"][t]:
            card.setdefault(int(ep["player_ids"][t]), int(np.argmax(ep["observations"][t][2:5])))
    acts = [int(ep["actions"][t]) for t in range(len(ep["valid"])) if ep["valid"][t]]
    return [card[0], card[1]] + acts


def _leduc_sequence(ep):
    # infostate tensor (leduc_poker.cc:170-192): player(2) . private card(6) . public card(6) . betting[2][4][2]
    card, public, seq = {}, None, []
    steps = [t for t in range(len(ep["valid"])) if ep["valid"][t]]
    for t in steps:
        o = ep["observations"][t]
        card.setdefault(int(ep["player_ids"][t]), int(np.argmax(o[2:8])))
        if public is None and o[8:14].any():
            public = int(np.argmax(o[8:14]))
    seq = [card[0], card[1]]
    dealt_public = False
    for t in steps:
        if not dealt_public and ep["observations"][t][8:14].any():
            seq.append(public)
            dealt_public = True
        seq.append(int(ep["actions"][t]))
    return seq


CASES = [("kuhn_poker", 5, _kuhn_sequence), ("leduc_poker", 10, _leduc_sequence)]


def reference_golden():
    import ref_lib
    out = {}
    for name, T, sequence in CASES:
        ref = ref_lib.ref_record_batched_trajectory(ref_lib.RefGame(name), B, seed=1234, T=T)
        d = Digest()
        seqs = []
        for b in range(B):
            ep = {k: v[b] for k, v in ref.items()}
            seqs.append([int(x) for x in sequence(ep)])
            d.add([ep[k] for k in FIELDS])
        out["trajectories/" + name] = {"sequences": seqs, "digest": d.hexdigest()}
    return out


@pytest.mark.parametrize("name,T,sequence", CASES)
def test_oracle_recorder_reproduces_reference_episodes(name, T, sequence):
    want = expected("trajectories/" + name)
    og = OracleGame(name)
    d = Digest()
    lengths = set()
    for forced in want["sequences"]:
        mine = oracle_record_trajectory(og.new_initial_state(), seed=0, lane=0, T=T, forced=forced)
        assert mine["length"] == int(mine["valid"].sum())
        assert sequence(mine) == forced          # the episode's tensors name the same chance outcomes and actions
        lengths.add(mine["length"])
        # player_policies of the uniform policy: 1/#legal on the legal actions; padding rows all ones (ResizeFields)
        la = mine["legal_actions"].astype(np.float64)
        mine["player_policies"] = np.where(mine["valid"][:, None] == 1, la / la.sum(-1, keepdims=True), 1.0)
        d.add([np.asarray(mine[k]) for k in FIELDS])
    assert len(want["sequences"]) == B and d.hexdigest() == want["digest"]
    assert len(lengths) > 1          # ragged batch: the padding convention was exercised


def test_oracle_recorder_is_a_legal_uniform_random_episode():
    """Sampling mode (the device recorder's stream): structural checks on every game."""
    for gs, T in [("tic_tac_toe", 9), ("connect_four", 42), ("breakthrough(rows=6,columns=6)", 120), ("hex(board_size=5)", 25),
                  ("go(board_size=5)", 50), ("kuhn_poker", 5), ("leduc_poker", 10)]:
        og = OracleGame(gs)
        for lane in range(20):
            tr = oracle_record_trajectory(og.new_initial_state(), seed=99, lane=lane, T=T)
            n = tr["length"]
            assert 0 < n <= T
            assert tr["valid"][:n].all() and not tr["valid"][n:].any()
            assert tr["next_is_terminal"].sum() == 1 and tr["next_is_terminal"][n - 1] == 1
            assert (tr["legal_actions"][n:] == 1).all() and not tr["observations"][n:].any()
            for t in range(n):
                assert tr["legal_actions"][t, tr["actions"][t]] == 1


def test_batched_trajectory_host_views_on_cpu_tensors():
    """Host logic of open_spiel_b200.BatchedTrajectory (bit-mask expansion, [B, T] views of time-major buffers, uniform
    player_policies) exercised on CPU tensors filled from oracle episodes."""
    import torch
    from open_spiel_b200.spiel import BatchedTrajectory
    og = OracleGame("connect_four")
    B, T, A = 16, 42, 7
    eps = [oracle_record_trajectory(og.new_initial_state(), seed=3, lane=i, T=T) for i in range(B)]
    legal = np.stack([e["legal_actions"] for e in eps])                       # [B, T, A]
    words = (legal.astype(np.int64) << np.arange(A)).sum(-1).astype(np.int32)  # bit a of word 0
    tm = {
        "observations": None,
        "legal_mask": torch.from_numpy(words.T.copy()).reshape(T, B, 1),
        "actions": torch.from_numpy(np.stack([e["actions"] for e in eps]).T.astype(np.int32).copy()),
        "player_ids": torch.from_numpy(np.stack([e["player_ids"] for e in eps]).T.astype(np.int8).copy()),
        "valid": torch.from_numpy(np.stack([e["valid"] for e in eps]).T.astype(np.uint8).copy()),
        "next_is_terminal": torch.from_numpy(np.stack([e["next_is_terminal"] for e in eps]).T.astype(np.uint8).copy()),
        "rewards": torch.from_numpy(np.stack([e["rewards"] for e in eps]).astype(np.float32)),
        "lengths": torch.tensor([e["length"] for e in eps], dtype=torch.int32),
    }
    tr = BatchedTrajectory(B, T, A, tm)
    assert tr.actions.shape == (B, T) and tr.legal_mask.shape == (B, T, 1)
    assert np.array_equal(tr.legal_actions().numpy(), legal)
    valid = np.stack([e["valid"] for e in eps])
    la = legal.astype(np.float64)
    want = np.where(valid[:, :, None] == 1, la / la.sum(-1, keepdims=True), 1.0)
    assert np.array_equal(tr.player_policies().numpy(), want)
    assert int(tr.valid.sum()) == int(tr.lengths.sum())

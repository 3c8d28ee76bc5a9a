"""GPU parity: every batched State function vs the CPU oracle, bit-exact, on seeded random games."""
import json
import os
import glob

import numpy as np
import pytest
import torch

import open_spiel_b200 as b2
from oracle_lib import OracleGame
from parity import lockstep, mask_words_to_lists

pytestmark = pytest.mark.gpu

GAMES = [
    ("tic_tac_toe", 512),
    ("connect_four", 512),
    ("connect_four(rows=4,columns=5,x_in_row=3)", 256),       # connect_four_test.cc:319-395 sizes
    ("connect_four(rows=5,columns=6)", 256),
    ("connect_four(rows=7,columns=8,x_in_row=5)", 256),
    ("connect_four(egocentric_obs_tensor=True)", 128),
    ("breakthrough", 256),
    ("breakthrough(rows=6,columns=6)", 128),
    ("breakthrough(rows=5,columns=4)", 128),
    ("hex", 128),
    ("hex(board_size=5)", 256),
    ("hex(num_cols=4,num_rows=3)", 128),
    ("hex(board_size=4,swap=True)", 256),
    ("hex(board_size=5,plain_obs_tensor=True)", 64),
    ("hex(num_cols=5,num_rows=3,plain_obs_tensor=True)", 64),
    ("go(board_size=9)", 96),
    ("go(board_size=5)", 256),
    ("go(board_size=7,komi=4.5)", 64),
    ("go(board_size=9,max_game_length=40)", 64),
    ("go(board_size=3,komi=0.5)", 256),
    ("go(board_size=4,komi=0.5)", 256),
    ("go(board_size=2,komi=0.5)", 128),
    ("havannah", 96),
    ("havannah(board_size=4)", 512),
    ("havannah(board_size=4,swap=True)", 512),
    ("havannah(board_size=2)", 64),
    ("y(board_size=9)", 512),
    ("y(board_size=11)", 128),
    ("y(board_size=2)", 64),
    ("othello", 512),
    ("mnk", 48),
    ("mnk(m=3,n=3,k=3)", 512),
    ("mnk(m=7,n=5,k=4)", 128),
    ("mnk(m=15,n=15,k=3)", 64),
    ("mnk(m=4,n=15,k=5)", 64),
    ("mnk(m=5,n=5,k=7)", 64),
    ("mnk(m=1,n=1,k=1)", 32),
    ("kuhn_poker", 512),
    ("kuhn_poker(players=3)", 512),
    ("kuhn_poker(players=5)", 256),
    ("leduc_poker", 1024),
    ("leduc_poker(players=3)", 1024),
    ("leduc_poker(players=4)", 256),
    ("leduc_poker(starting_player=1)", 256),
]
# the same games again at several blocks of the ILP kernels with a ragged last warp: 2085 = 2 * (256 * 4) + 37 lanes at
# ILP 4, 1061 = 2 * (256 * 2) + 37 at ILP 2
MULTI_BLOCK = [
    ("tic_tac_toe", 2085),
    ("connect_four", 2085),
    ("kuhn_poker", 2085),
    ("leduc_poker", 2085),
    ("breakthrough", 1061),
    ("othello", 1061),
]
INFO_STATE = {"kuhn_poker", "kuhn_poker(players=3)", "kuhn_poker(players=5)", "leduc_poker", "leduc_poker(starting_player=1)",
              "leduc_poker(players=3)", "leduc_poker(players=4)"}


@pytest.mark.parametrize("game_string,lanes", GAMES + MULTI_BLOCK,
                         ids=[g for g, _ in GAMES] + ["%s-%d" % (g, n) for g, n in MULTI_BLOCK])
def test_lockstep_random_games(game_string, lanes):
    steps = lockstep(game_string, n_lanes=lanes, seed=1234, check_info_state=game_string in INFO_STATE)
    assert steps >= lanes


def test_illegal_and_noop_actions_connect_four():
    g = b2.load_game("connect_four")
    b = g.new_batch(8)
    dev = b._dev
    # fill column 0 on lanes 0..3 (6 stones), then a 7th drop must be rejected and leave the lane intact
    for _ in range(6):
        b.apply_actions(torch.tensor([0, 0, 0, 0, -1, -1, -1, -1], dtype=torch.int32, device=dev))
    assert b.error_count()[0] == 0
    before = [b.state_blob(i) for i in range(8)]
    b.apply_actions(torch.tensor([0, 7, -2, 1, -1, -1, -1, -1], dtype=torch.int32, device=dev))
    cnt, first = b.error_count()
    assert cnt == 3 and first == 0
    after = [b.state_blob(i) for i in range(8)]
    assert before[0] == after[0] and before[1] == after[1] and before[2] == after[2]
    assert before[3] != after[3]
    assert before[4:] == after[4:]          # -1 lanes untouched
    b.reset()
    assert b.error_count()[0] == 0


def test_actions_on_terminal_states_are_rejected():
    # connect_four_test.cc:38-58 FastLoss: 3,3,4,4,2,2,1 -> x wins
    g = b2.load_game("connect_four")
    b = g.new_batch(4)
    for a in [3, 3, 4, 4, 2, 2, 1]:
        b.apply_actions(torch.full((4,), a, dtype=torch.int32, device=b._dev))
    cur, term, rets = b.status()
    assert term.tolist() == [1] * 4 and cur.tolist() == [-4] * 4
    assert rets.tolist() == [[1.0, -1.0]] * 4
    assert b.legal_actions_mask_words().flatten().tolist() == [0] * 4
    b.apply_actions(torch.full((4,), 0, dtype=torch.int32, device=b._dev))
    assert b.error_count()[0] == 4


def test_scalar_state_adapter_reads_like_pyspiel():
    game = b2.load_game("tic_tac_toe")
    state = game.new_initial_state()
    assert state.current_player() == 0 and not state.is_terminal()
    assert state.legal_actions() == list(range(9))
    state.apply_action(4)
    assert state.legal_actions() == [0, 1, 2, 3, 5, 6, 7, 8]
    clone = state.clone()
    state.apply_action(0)
    assert clone.history() == [4] and state.history() == [4, 0]
    assert clone.legal_actions() == [0, 1, 2, 3, 5, 6, 7, 8]
    with pytest.raises(b2.SpielError):
        state.apply_action(4)
    for a in [3, 1, 5]:       # x: 4,3,5 -> middle row
        state.apply_action(a)
    assert state.is_terminal() and state.returns() == [1.0, -1.0]
    assert state.current_player() == -4 and state.legal_actions() == []
    assert state.serialize() == "4\n0\n3\n1\n5\n"


GOLD = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "playthroughs", "*.json")))


@pytest.mark.parametrize("path", GOLD, ids=[os.path.basename(p)[:-5] for p in GOLD])
def test_device_replays_reference_playthrough(path):
    """The reference's own golden traces (integration_tests/playthrough_test.py:73-98), replayed on the GPU."""
    gold = json.load(open(path, encoding="utf-8"))
    try:
        game = b2.load_game(gold["game"])
        state = game.new_initial_state()
    except b2.SpielError as e:
        pytest.skip(str(e))
    hdr = gold["header"]
    assert game.num_distinct_actions() == int(hdr["NumDistinctActions"])
    assert game.max_game_length() == int(hdr["MaxGameLength"])
    for k, g in enumerate(gold["states"]):
        if g["detailed"]:
            assert state.is_terminal() == g["is_terminal"]
            assert state.current_player() == g["current_player"]
            assert state.history() == g["history"]
            if "legal_actions" in g:
                assert state.legal_actions() == g["legal_actions"]
            if "returns" in g:
                r = state.returns()
                assert r == g["returns"]
                assert [np.signbit(x) for x in r] == [t.startswith("-") for t in g["returns_text"]]
            for name, vals in g["tensors"].items():
                p = int(name[name.index("(") + 1:name.index(")")])
                t = state.observation_tensor(p) if name.startswith("Observation") else state.information_state_tensor(p)
                np.testing.assert_array_equal(t, np.array(vals, dtype=np.float32), err_msg=name)
        if k < len(gold["actions"]):
            state.apply_action(gold["actions"][k])
    assert state.is_terminal()


def test_rollout_matches_oracle_given_same_random_stream():
    """b2s_rollout = uniform-random playout; the oracle replays it with the same Philox words."""
    from philox_ref import philox_uniform
    for gs in ["connect_four", "tic_tac_toe", "breakthrough", "hex(board_size=5)", "go(board_size=5)", "kuhn_poker",
               "leduc_poker", "mnk(m=6,n=6,k=4)", "othello", "y(board_size=7)", "havannah(board_size=4)"]:
        game = b2.load_game(gs)
        n = 256
        b = game.new_batch(n)
        rets, plies = b.rollout(seed=0x5EED, lane_offset=1000)
        rets, plies = rets.cpu().numpy(), plies.cpu().numpy()
        og = OracleGame(gs)
        for i in range(n):
            st = og.new_initial_state()
            ply = 0
            while not st.is_terminal():
                la, cand = st.legal_actions(), st.rollout_candidates()
                retry = 0
                while True:          # uniform over legal actions by rejection from the candidate list
                    a = cand[philox_uniform(0x5EED, 1000 + i, ply + 4096 * retry, len(cand))]
                    if a in la:
                        break
                    retry += 1
                st.apply_action(a)
                ply += 1
            assert ply == plies[i], (gs, i)
            assert st.returns() == rets[i].tolist(), (gs, i)
        _, term, rets2 = b.status()
        assert term.all() and np.array_equal(rets2.cpu().numpy(), rets)


def test_full_size_properties_connect_four():
    """BASELINE config 2 size (1M lanes): size-independent properties."""
    game = b2.load_game("connect_four")
    n = 1 << 20
    b = game.new_batch(n)
    rets, plies = b.rollout(seed=7)
    cur, term, rets2 = b.status()
    assert bool(term.all()) and bool((cur == -4).all())
    assert torch.equal(rets, rets2)
    assert bool((rets.sum(dim=1) == 0).all())                       # zero-sum
    assert int(plies.min()) >= 7 and int(plies.max()) <= 42         # shortest win is 7 plies
    draws = (rets[:, 0] == 0)
    assert bool((plies[draws] == 42).all())                         # draws only on a full board
    assert int(b.legal_actions_mask_words().abs().sum()) == 0
    # a deterministic replay of the same seed gives bit-identical states
    b2_ = game.new_batch(n)
    b2_.rollout(seed=7)
    assert torch.equal(b.observation_tensor(0, n=4096), b2_.observation_tensor(0, n=4096))
    # observation planes partition the board: exactly one plane set per cell
    obs = b.observation_tensor(0, n=65536).reshape(-1, 3, 42)
    assert bool((obs.sum(dim=1) == 1).all())


def test_host_buffer_step_equals_device_step_across_chunks():
    """b2s_step_fused_host uploads / steps / downloads in overlapping chunks: outputs must equal the device-buffer call on
    an identical batch, and a rejected action must be reported with its batch lane (not its lane within a chunk)."""
    n = (1 << 19) + 777                                       # > 2^18: chunked path, ragged last chunk
    game = b2.load_game("connect_four")
    a, b = game.new_batch(n), game.new_batch(n)
    g = torch.Generator(device="cpu").manual_seed(5)
    mask_h = torch.empty((n, 1), dtype=torch.int32).pin_memory()
    term_h = torch.empty((n,), dtype=torch.uint8).pin_memory()
    rets_h = torch.empty((n, 2), dtype=torch.float32).pin_memory()
    for ply in range(12):
        acts = torch.randint(0, 7, (n,), generator=g, dtype=torch.int32)    # early plies: every column is legal
        acts_h = acts.pin_memory()
        m, t, r = a.step(acts.to(a._dev))
        b.step_host(acts_h, mask_h, term_h, rets_h)
        if ply < 6:
            assert a.error_count()[0] == 0 and b.error_count()[0] == 0
        assert torch.equal(m.cpu().reshape(-1), mask_h.reshape(-1))
        assert torch.equal(t.cpu(), term_h) and torch.equal(r.cpu(), rets_h)
    # one illegal action far from lane 0: column 0 six more times fills it, the seventh drop is rejected
    c = game.new_batch(n)
    bad_lane = 3 * (1 << 17) + 12345
    acts_h = torch.full((n,), -1, dtype=torch.int32).pin_memory()
    acts_h[bad_lane] = 0
    for _ in range(7):
        c.step_host(acts_h, mask_h, term_h, rets_h)
    cnt, first = c.error_count()
    assert cnt >= 1 and first == bad_lane


def test_host_step_graph_replay_equals_stream_path():
    """With pinned buffers and n >= 65536 b2s_step_fused_host replays a captured CUDA graph of its chunked upload -> kernel ->
    download pipeline, and the byte-wide entry reads / writes the pinned buffers from the kernel itself (zero copy); pageable
    buffers take the plain stream path.  Same inputs, same outputs, call after call."""
    from open_spiel_b200 import _lib
    n = (1 << 17) + 333
    game = b2.load_game("connect_four")
    a, b, c = game.new_batch(n), game.new_batch(n), game.new_batch(n)
    g = torch.Generator(device="cpu").manual_seed(11)
    pin = lambda t: t.pin_memory()   # noqa: E731
    acts_p, acts_u = pin(torch.empty((n,), dtype=torch.int32)), torch.empty((n,), dtype=torch.int32)
    acts8_p = pin(torch.empty((n,), dtype=torch.uint8))
    mask_p, term_p, rets_p = pin(torch.empty((n, 1), dtype=torch.int32)), pin(torch.empty((n,), dtype=torch.uint8)), pin(torch.empty((n, 2), dtype=torch.float32))
    mask_u, term_u, rets_u = torch.empty((n, 1), dtype=torch.int32), torch.empty((n,), dtype=torch.uint8), torch.empty((n, 2), dtype=torch.float32)
    status_p = pin(torch.empty((n,), dtype=torch.uint8))
    before, zc_before = _lib.lib().b2s_host_graph_launches(), _lib.lib().b2s_host_zero_copy_steps()
    for ply in range(10):
        acts = torch.randint(0, 7, (n,), generator=g, dtype=torch.int32)
        acts_p.copy_(acts); acts_u.copy_(acts); acts8_p.copy_(acts.to(torch.uint8))
        a.step_host(acts_p, mask_p, term_p, rets_p)                 # pinned: graph
        b.step_host(acts_u, mask_u, term_u, rets_u)                 # pageable: streams
        c.step_host_compact(acts8_p, status_p)                      # pinned, byte-wide: zero copy
        assert torch.equal(mask_p, mask_u) and torch.equal(term_p, term_u) and torch.equal(rets_p, rets_u)
        t = term_u.bool()
        assert torch.equal(status_p >> 7, term_u)
        assert torch.equal((status_p & 0x7F)[~t], mask_u[:, 0].to(torch.uint8)[~t])
    assert a.error_count()[0] == b.error_count()[0] == c.error_count()[0]
    replays = _lib.lib().b2s_host_graph_launches() - before
    zero_copy = _lib.lib().b2s_host_zero_copy_steps() - zc_before
    print("host-step graph replays:", replays, "zero-copy steps:", zero_copy)
    assert replays in (0, 10)          # 0 only when the capture is not supported on this driver (the library then stays on the stream path)
    assert zero_copy in (0, 10)        # 0 only when pinned memory is not device-mapped here
    # ragged sizes and the no-op byte through the zero-copy kernel, against the device-buffer step
    for m in (4096 + 5, 70001):
        d, e = game.new_batch(m), game.new_batch(m)
        a8 = torch.randint(0, 7, (m,), generator=g, dtype=torch.int32)
        a8[::7] = -1                                              # untouched lanes
        a8_p = pin(torch.where(a8 < 0, torch.full_like(a8, 255), a8).to(torch.uint8))
        st_p = pin(torch.zeros((m,), dtype=torch.uint8))
        mk, tm, _ = d.step(a8.to(d._dev))
        e.step_host_compact(a8_p, st_p)
        assert torch.equal(st_p >> 7, tm.cpu())
        live = ~tm.cpu().bool()
        assert torch.equal((st_p & 0x7F)[live], mk.cpu()[:, 0].to(torch.uint8)[live])
        assert d.error_count()[0] == e.error_count()[0]

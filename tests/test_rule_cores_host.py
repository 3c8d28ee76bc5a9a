"""CPU: the PRODUCT's rule cores (open_spiel_b200/csrc/rules_*.cuh), compiled for the host by tests/host_emul (test
infrastructure: the library itself has no CPU path), played lock-step against the oracle: current player, terminal flag,
returns (sign of zero included), legal-action mask, observation and information-state tensors after every move of
random games, for every game and parameter variant the device supports.  This checks the bit-twiddling the CUDA kernels
are built from without a GPU; launch geometry and memory staging are covered by the -m gpu tests."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import open_spiel_b200 as b2
from open_spiel_b200._lib import GameInfo
from oracle_lib import OracleGame

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_emul")


def _lib():
    so = os.path.join(HERE, "libemul.so")
    if not os.path.exists(so):
        subprocess.run(["make", "-C", HERE], capture_output=True)
    if not os.path.exists(so):
        pytest.skip("host emulation library not built (needs g++ and the CUDA headers)")
    L = C.CDLL(so)
    L.emu_create.restype = C.c_void_p
    L.emu_create.argtypes = [C.c_int, C.c_void_p, C.c_longlong]
    L.emu_last_error.restype = C.c_char_p
    for name, args in (("emu_destroy", [C.c_void_p]), ("emu_info", [C.c_void_p, C.c_void_p]),
                       ("emu_reset", [C.c_void_p, C.c_longlong]), ("emu_apply", [C.c_void_p, C.c_void_p, C.c_longlong]),
                       ("emu_legal_mask", [C.c_void_p, C.c_void_p, C.c_longlong]),
                       ("emu_status", [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong]),
                       ("emu_observation", [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_longlong])):
        getattr(L, name).argtypes = args
    L.emu_error_count.restype = C.c_longlong
    L.emu_error_count.argtypes = [C.c_void_p]
    L.emu_rollout.argtypes = [C.c_void_p, C.c_ulonglong, C.c_longlong, C.c_void_p, C.c_void_p, C.c_longlong]
    L.emu_mcts.argtypes = [C.c_void_p, C.c_longlong, C.c_void_p] + [C.c_void_p] * 5
    return L


class Emu:
    def __init__(self, game_string, n):
        self.L = _lib()
        g = b2.load_game(game_string)                       # parameter parsing only; no device is touched
        self.h = self.L.emu_create(g._gid, C.byref(g._cparams), n)
        assert self.h, self.L.emu_last_error()
        self.info = GameInfo()
        self.L.emu_info(self.h, C.byref(self.info))
        self.n = n
        self.L.emu_reset(self.h, n)

    def __del__(self):
        try:
            self.L.emu_destroy(self.h)
        except Exception:
            pass

    def apply(self, actions):
        a = np.ascontiguousarray(actions, dtype=np.int32)
        self.L.emu_apply(self.h, a.ctypes.data, self.n)

    def legal(self):
        W = self.info.mask_words
        out = np.zeros((self.n, W), dtype=np.uint32)
        self.L.emu_legal_mask(self.h, out.ctypes.data, self.n)
        width = max(self.info.num_distinct_actions, self.info.max_chance_outcomes)
        bits = ((out[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1).reshape(self.n, -1)[:, :width]
        return [np.nonzero(r)[0].tolist() for r in bits]

    def status(self):
        cur = np.zeros(self.n, dtype=np.int8)
        term = np.zeros(self.n, dtype=np.uint8)
        rets = np.zeros((self.n, self.info.num_players), dtype=np.float32)
        self.L.emu_status(self.h, cur.ctypes.data, term.ctypes.data, rets.ctypes.data, self.n)
        return cur, term, rets

    def tensor(self, player, which):
        size = self.info.observation_tensor_size if which == 0 else self.info.information_state_tensor_size
        out = np.zeros((self.n, size), dtype=np.float32)
        assert self.L.emu_observation(self.h, player, which, out.ctypes.data, self.n) == 0
        return out

    def errors(self):
        return self.L.emu_error_count(self.h)

    def rollout(self, seed, lane_offset=0):
        rets = np.zeros((self.n, self.info.num_players), dtype=np.float32)
        plies = np.zeros(self.n, dtype=np.int32)
        self.L.emu_rollout(self.h, seed, lane_offset, rets.ctypes.data, plies.ctypes.data, self.n)
        return rets, plies

    def mcts(self, sims, uct_c=2.0, n_rollouts=1, solve=True, seed=0, offset=0, puct=False, max_nodes=0, budget=0):
        """max_nodes: physical arena nodes over all trees (0 = derived); budget: MCTSBot::max_nodes_ per tree (GC)."""
        from open_spiel_b200._lib import MctsConfig
        A = self.info.num_distinct_actions
        self.gc_runs = np.zeros(self.n, dtype=np.int32)
        cfg = MctsConfig(sims, n_rollouts, int(solve), int(puct), uct_c, seed, offset, max_nodes, budget, 0.0, self.gc_runs.ctypes.data)
        visits = np.zeros((self.n, A), dtype=np.int32)
        reward = np.zeros((self.n, A), dtype=np.float64)
        outcome = np.zeros((self.n, A), dtype=np.float32)
        best = np.zeros(self.n, dtype=np.int32)
        ran = np.zeros(self.n, dtype=np.int32)
        rc = self.L.emu_mcts(self.h, self.n, C.byref(cfg), visits.ctypes.data, reward.ctypes.data, outcome.ctypes.data,
                             best.ctypes.data, ran.ctypes.data)
        assert rc == 0
        return visits, reward, outcome, best, ran


GAMES = [
    ("tic_tac_toe", 64), ("connect_four", 64), ("connect_four(rows=4,columns=5,x_in_row=3)", 48),
    ("connect_four(rows=7,columns=8,x_in_row=5)", 32), ("connect_four(egocentric_obs_tensor=True)", 32),
    ("breakthrough", 24), ("breakthrough(rows=6,columns=6)", 32), ("breakthrough(rows=5,columns=4)", 32),
    ("hex", 16), ("hex(board_size=5)", 48), ("hex(num_cols=3,num_rows=5)", 32), ("hex(board_size=4,swap=True)", 48),
    ("hex(board_size=5,plain_obs_tensor=True)", 24),
    ("go(board_size=9)", 12), ("go(board_size=5)", 32), ("go(board_size=3,komi=0.5)", 48), ("go(board_size=7,komi=4.5)", 16),
    ("go(board_size=5,max_game_length=30)", 24),
    ("kuhn_poker", 128), ("kuhn_poker(players=3)", 192), ("kuhn_poker(players=4)", 128), ("kuhn_poker(players=5)", 128),
    ("havannah", 48), ("havannah(board_size=4)", 256), ("havannah(board_size=4,swap=True)", 256), ("havannah(board_size=6)", 64),
    ("havannah(board_size=2)", 64), ("havannah(board_size=3,swap=True)", 128), ("havannah(board_size=1)", 4),
    ("y(board_size=9)", 128), ("y(board_size=11)", 64), ("y(board_size=1)", 8), ("y(board_size=2)", 32), ("y(board_size=4)", 128),
    ("othello", 96), ("mnk", 24), ("mnk(m=3,n=3,k=3)", 128), ("mnk(m=7,n=5,k=4)", 64), ("mnk(m=15,n=15,k=3)", 32), ("mnk(m=4,n=15,k=5)", 32),
    ("mnk(m=1,n=1,k=1)", 8), ("mnk(m=5,n=5,k=7)", 32),
    ("leduc_poker", 128), ("leduc_poker(starting_player=1)", 64), ("leduc_poker(players=3)", 256),
    ("leduc_poker(players=3,starting_player=2)", 128), ("leduc_poker(players=4)", 128),
]


@pytest.mark.parametrize("gs,n", GAMES, ids=[g for g, _ in GAMES])
def test_rule_core_lockstep_vs_oracle(gs, n):
    _lockstep(gs, n, OracleGame)


REF_GAMES = [(g, max(8, k // 3)) for g, k in GAMES]


@pytest.mark.parametrize("gs,n", REF_GAMES, ids=[g for g, _ in GAMES])
def test_rule_core_lockstep_vs_unmodified_reference(gs, n):
    """The same lock-step play with the UNMODIFIED reference as the checker: the code the CUDA kernels are built from
    against open_spiel's own State classes, in the CPU suite.  The reference's side is stored (tests/reference_golden.py):
    a digest of everything _lockstep compares, along the same games."""
    from reference_golden import Digest, expected
    want = expected("rule_cores/" + gs)
    emu = Emu(gs, n)
    info = emu.info
    P, has_info = info.num_players, want["has_info"]
    rng = np.random.RandomState(sum(map(ord, gs)) % 997)
    d = Digest([info.num_distinct_actions, info.max_game_length, info.num_players, info.observation_tensor_size])
    for ply in range(info.max_game_length + 8):
        cur, term, rets = emu.status()
        legal = emu.legal()
        obs = [emu.tensor(p, 0) for p in range(P)]
        ist = [emu.tensor(p, 1) for p in range(P)] if has_info else None
        actions = np.full(n, -1, dtype=np.int32)
        for i in range(n):
            _record(d, cur[i], term[i], legal[i], rets[i].tolist(), [o[i] for o in obs], ist and [t[i] for t in ist])
            if not term[i]:
                actions[i] = legal[i][rng.randint(len(legal[i]))]
        if (actions < 0).all():
            break
        emu.apply(actions)
        assert emu.errors() == 0
    else:
        raise AssertionError("games did not end")
    assert d.hexdigest() == want["digest"]


def _record(d, cur, term, legal, rets, obs, ist):
    d.add(int(cur), bool(term), legal, [float(x).hex() for x in rets], obs, ist)


def reference_golden():
    """The reference's side of test_rule_core_lockstep_vs_unmodified_reference: its states played the same way."""
    import ref_lib
    from reference_golden import Digest
    out = {}
    for gs, n in REF_GAMES:
        g = ref_lib.RefGame(gs)
        rng = np.random.RandomState(sum(map(ord, gs)) % 997)
        has_info = g.information_state_tensor_size > 0
        P = g.num_players
        d = Digest([g.num_distinct_actions, g.max_game_length, g.num_players, g.observation_tensor_size])
        states = [g.new_initial_state() for _ in range(n)]
        while True:
            actions = []
            for st in states:
                _record(d, st.current_player(), st.is_terminal(), st.legal_actions(), st.returns(),
                        [st.observation_tensor(p) for p in range(P)],
                        [st.information_state_tensor(p) for p in range(P)] if has_info else None)
                la = st.legal_actions()
                actions.append(None if st.is_terminal() else la[rng.randint(len(la))])
            if all(a is None for a in actions):
                break
            for st, a in zip(states, actions):
                if a is not None:
                    st.apply_action(a)
        out["rule_cores/" + gs] = {"digest": d.hexdigest(), "has_info": has_info}
    return out


def _lockstep(gs, n, checker):
    rng = np.random.RandomState(sum(map(ord, gs)) % 997)
    og = checker(gs)
    emu = Emu(gs, n)
    info = emu.info
    assert (info.num_distinct_actions, info.max_game_length, info.num_players) == (og.num_distinct_actions, og.max_game_length,
                                                                                  og.num_players)
    assert info.observation_tensor_size == og.observation_tensor_size
    has_info = og.information_state_tensor_size > 0
    states = [og.new_initial_state() for _ in range(n)]
    P = og.num_players
    for ply in range(og.max_game_length + 8):
        cur, term, rets = emu.status()
        legal = emu.legal()
        obs = [emu.tensor(p, 0) for p in range(P)]
        ist = [emu.tensor(p, 1) for p in range(P)] if has_info else None
        actions = np.full(n, -1, dtype=np.int32)
        alive = 0
        for i, st in enumerate(states):
            assert int(cur[i]) == st.current_player(), (gs, i, ply)
            assert bool(term[i]) == st.is_terminal(), (gs, i, ply)
            ola = st.legal_actions()
            assert legal[i] == ola, (gs, i, ply, legal[i], ola, st.to_string())
            want = np.array(st.returns())
            assert rets[i].tolist() == want.tolist() and np.array_equal(np.signbit(rets[i]), np.signbit(want)), (gs, i, ply)
            for p in range(P):
                np.testing.assert_array_equal(obs[p][i], st.observation_tensor(p), err_msg="%s lane %d ply %d" % (gs, i, ply))
                if has_info:
                    np.testing.assert_array_equal(ist[p][i], st.information_state_tensor(p))
            if not st.is_terminal():
                a = ola[rng.randint(len(ola))]
                actions[i] = a
                st.apply_action(a)
                alive += 1
        if alive == 0:
            break
        emu.apply(actions)
        assert emu.errors() == 0
    else:
        raise AssertionError("games did not end")


def test_rule_core_rejects_illegal_and_post_terminal_actions():
    emu = Emu("connect_four", 4)
    for _ in range(6):
        emu.apply([0, -1, -1, -1])                   # fill column 0 of lane 0
    assert emu.errors() == 0
    before = emu.legal()
    emu.apply([0, 9, -2, -1])                        # full column, out of range, negative: three rejected lanes
    assert emu.errors() == 3 and emu.legal() == before
    ttt = Emu("tic_tac_toe", 1)
    for a in (0, 3, 1, 4, 2):                        # x wins on the top row
        ttt.apply([a])
    assert ttt.status()[1][0] == 1 and ttt.errors() == 0
    ttt.apply([5])                                   # acting on a terminal state is rejected, state unchanged
    assert ttt.errors() == 1 and ttt.status()[2][0].tolist() == [1.0, -1.0]


@pytest.mark.parametrize("gs", ["connect_four", "tic_tac_toe", "breakthrough", "breakthrough(rows=6,columns=6)", "hex(board_size=5)",
                                "go(board_size=5)", "go(board_size=9)", "kuhn_poker", "leduc_poker", "mnk(m=6,n=6,k=4)", "othello", "y(board_size=7)", "havannah(board_size=4)"])
def test_playout_step_matches_oracle_given_same_random_stream(gs):
    """common.cuh playout_step (legal-mask draw; candidate rejection sampling for go and breakthrough) on the host vs the
    oracle replaying the same Philox words — the CPU twin of the GPU test of b2s_rollout."""
    from philox_ref import philox_uniform
    n = 24 if "9" in gs else 64
    emu = Emu(gs, n)
    rets, plies = emu.rollout(0x5EED, 1000)
    og = OracleGame(gs)
    for i in range(n):
        st = og.new_initial_state()
        ply = 0
        while not st.is_terminal():
            la, cand = st.legal_actions(), st.rollout_candidates()
            retry = 0
            while True:
                a = cand[philox_uniform(0x5EED, 1000 + i, ply + 4096 * retry, len(cand))]
                if a in la:
                    break
                retry += 1
            st.apply_action(a)
            ply += 1
        assert ply == plies[i] and st.returns() == rets[i].tolist(), (gs, i)
    assert emu.status()[1].all()


MCTS_CASES = [("tic_tac_toe", 16, 3, 300, 2, True, False), ("connect_four", 12, 8, 200, 1, True, False),
              ("connect_four(rows=4,columns=5,x_in_row=3)", 12, 5, 300, 1, True, True),
              ("breakthrough(rows=6,columns=6)", 8, 8, 100, 1, True, False), ("hex(board_size=5)", 12, 6, 150, 1, True, False),
              ("hex(board_size=4,swap=True)", 8, 2, 150, 1, True, True), ("go(board_size=5)", 12, 8, 100, 1, True, False),
              ("go(board_size=9)", 6, 20, 30, 1, True, False),
              # tiny boards: positional superko decides playouts, so the root's hash history must reach the work lanes
              ("go(board_size=2)", 6, 5, 80, 2, False, True), ("go(board_size=3)", 6, 5, 80, 2, False, True),
              ("go(board_size=2)", 6, 12, 60, 1, True, True),
              # n_rollouts not a power of two: 24-byte nodes with the reference's double accumulator
              ("tic_tac_toe", 8, 2, 200, 3, True, False), ("connect_four", 6, 4, 150, 5, False, True),
              # node budget + garbage collection (mcts.cc:441-482): (.., budget) as an 8th field
              ("connect_four", 6, 4, 1500, 1, False, False, 300), ("tic_tac_toe", 6, 1, 1200, 2, True, False, 120),
              ("hex(board_size=4)", 6, 2, 1500, 1, True, True, 400), ("go(board_size=5)", 4, 4, 600, 1, True, False, 500),
              ("breakthrough(rows=5,columns=4)", 4, 3, 800, 1, False, False, 250),
              # next-tier games (SURVEY 8 f.4): pass moves in the tree (othello), wide boards (mnk)
              ("othello", 8, 30, 120, 1, True, False), ("othello", 6, 56, 400, 1, True, True), ("othello", 4, 10, 900, 1, False, False, 300),
              ("havannah(board_size=3)", 8, 4, 300, 1, True, False), ("havannah(board_size=4,swap=True)", 6, 10, 150, 1, True, True),
              ("havannah(board_size=3)", 6, 2, 1200, 1, True, False, 300), ("havannah", 4, 30, 40, 1, True, False),
              ("y(board_size=5)", 8, 4, 300, 1, True, False), ("y(board_size=9)", 6, 12, 100, 1, True, True),
              ("y(board_size=4)", 6, 2, 1200, 1, True, False, 300),
              ("mnk(m=5,n=5,k=4)", 8, 6, 200, 1, True, False), ("mnk", 4, 10, 60, 1, True, True),
              ("mnk(m=4,n=4,k=3)", 6, 2, 1200, 2, True, False, 350)]


@pytest.mark.parametrize("case", MCTS_CASES, ids=["%s-%d-%d%s" % (c[0], c[3], c[4], "-gc" if len(c) > 7 else "") for c in MCTS_CASES])
def test_mcts_kernel_body_on_host_equals_oracle(case):
    gs, n, prefix, sims, nroll, solve, puct = case[:7]
    budget = case[7] if len(case) > 7 else 0
    """The body of the k_mcts kernel (mcts.cuh), executed on the host one tree at a time, vs the oracle's MCTS on the same
    Philox stream: visit counts, total rewards (exact doubles), proven outcomes, BestChild, simulations run."""
    import math
    from oracle_lib import oracle_mcts
    rng = np.random.RandomState(len(gs) + sims)
    og = OracleGame(gs)
    emu = Emu(gs, n)
    states = [og.new_initial_state() for _ in range(n)]
    ks = rng.randint(0, prefix + 1, size=n)
    for t in range(prefix):
        acts = np.full(n, -1, dtype=np.int32)
        for i, st in enumerate(states):
            if t < ks[i] and not st.is_terminal():
                la = st.legal_actions()
                a = la[rng.randint(len(la))]
                nxt = st.clone()
                nxt.apply_action(a)
                if nxt.is_terminal():
                    continue
                states[i] = nxt
                acts[i] = a
        emu.apply(acts)
    assert emu.errors() == 0
    visits, reward, outcome, best, ran = emu.mcts(sims, 2.0, nroll, solve, seed=0xC0FFEE, offset=17, puct=puct, budget=budget)
    assert emu.errors() == 0
    collections = 0
    for i, st in enumerate(states):
        o = oracle_mcts(st, 2.0, sims, nroll, solve, 0xC0FFEE, tree_index=i + 17, puct=puct, max_nodes=budget or 1)
        assert ran[i] == o["sims_run"], (gs, i)
        assert emu.gc_runs[i] == o["gc_runs"], (gs, i)
        collections += o["gc_runs"]
        for a, v, r, oc in o["children"]:
            assert visits[i, a] == v and reward[i, a] == r, (gs, i, a)
            assert (math.isnan(oc) and math.isnan(outcome[i, a])) or outcome[i, a] == oc, (gs, i, a)
        assert int(visits[i].sum()) == sum(v for _, v, _, _ in o["children"])
        assert best[i] == o["best_action"], (gs, i)
    if budget:
        assert collections >= n, "the budget must actually trigger garbage collections in this case"


def _sweep_variants():
    v = []
    for r, c, x in [(4, 4, 3), (4, 9, 4), (5, 6, 4), (6, 7, 5), (7, 7, 4), (7, 8, 4), (8, 7, 5), (6, 9, 5), (5, 4, 3)]:
        v.append("connect_four(rows=%d,columns=%d,x_in_row=%d)" % (r, c, x))
    for r, c in [(3, 3), (4, 2), (4, 8), (5, 5), (6, 3), (7, 7), (8, 2), (8, 7), (3, 8)]:
        v.append("breakthrough(rows=%d,columns=%d)" % (r, c))
    for r, c in [(2, 2), (2, 7), (3, 11), (7, 2), (11, 3), (6, 6), (9, 10), (11, 11)]:
        v.append("hex(num_rows=%d,num_cols=%d)" % (r, c))
    for r, c in [(2, 2), (3, 2), (5, 3), (6, 6), (8, 5), (9, 9)]:          # swap: rows >= cols (see the test below)
        v.append("hex(num_rows=%d,num_cols=%d,swap=True)" % (r, c))
    for bs, komi in [(2, 0.5), (3, 7.5), (4, 0.0), (6, 5.5), (7, 7.5), (8, 0.5), (9, 0.0)]:
        v.append("go(board_size=%d,komi=%s)" % (bs, komi))
    v += ["go(board_size=4,max_game_length=12)", "go(board_size=9,max_game_length=40)"]
    # next-tier games (SURVEY 8 f.4)
    for m, n, k in [(1, 5, 2), (2, 2, 2), (3, 15, 3), (15, 3, 3), (6, 6, 6), (9, 4, 4), (12, 13, 5), (15, 15, 15), (8, 8, 9)]:
        v.append("mnk(m=%d,n=%d,k=%d)" % (m, n, k))
    for bs in (1, 2, 3, 5, 6, 7, 8, 10, 11):
        v.append("y(board_size=%d)" % bs)
    for bs, swap in [(1, True), (2, True), (3, False), (5, False), (5, True), (6, True), (7, False), (8, True)]:
        v.append("havannah(board_size=%d%s)" % (bs, ",swap=True" if swap else ""))
    v += ["kuhn_poker(players=2)", "kuhn_poker(players=4)", "leduc_poker(players=4,starting_player=3)", "leduc_poker(players=3,starting_player=1)"]
    return v


@pytest.mark.parametrize("gs", _sweep_variants())
def test_rule_core_parameter_sweep(gs):
    """A committed sample of the 220-variant parameter fuzz run during development (0 mismatches)."""
    test_rule_core_lockstep_vs_oracle(gs, 6 if gs.startswith("go") else 10)


def test_hex_swap_on_wide_boards_is_reference_undefined_behaviour():
    """hex.cc:238 mirrors the first stone to cell c * num_cols + r without a bounds check: with more columns than rows that
    index can lie outside the board (undefined behaviour in the reference).  The oracle reports it as an error instead of
    writing out of bounds; parity is only defined — and checked above — for swap with rows >= cols."""
    with pytest.raises(b2.SpielError):                  # the device path refuses the configuration outright
        b2.load_game("hex(num_rows=2,num_cols=3,swap=True)")
    b2.load_game("hex(num_rows=3,num_cols=2,swap=True)")  # rows >= cols is well defined and supported
    st = OracleGame("hex(num_rows=2,num_cols=3,swap=True)").new_initial_state()
    st.apply_action(5)                                   # r = 1, c = 2 -> mirrored cell 2 * 3 + 1 = 7 >= 6
    with pytest.raises(RuntimeError):
        st.apply_action(6)                               # the swap action


def _havannah_lines(size):
    """Hand-built havannah games (actions = x + y * diameter) with a known end: (moves of player 0, moves of player 1, winner)."""
    d = 2 * size - 1
    c = lambda x, y: x + y * d   # noqa: E731
    far = [c(1, 1), c(5, 5), c(1, 2), c(5, 4), c(2, 1), c(4, 5)]                  # scattered, never connected to anything decisive
    ring = [c(2, 2), c(3, 2), c(4, 3), c(4, 4), c(3, 4), c(2, 3)]                  # the six neighbours of (3, 3): a ring
    bridge = [c(0, 0), c(1, 1), c(2, 2), c(3, 3), c(4, 4), c(5, 5), c(6, 6)]       # corner (0,0) to corner (6,6) along the diagonal
    fork = [c(1, 0), c(1, 1), c(1, 2), c(1, 3), c(0, 2), c(2, 3), c(3, 4), c(3, 5), c(3, 6)]   # touches edges 0, 5 and 3/4
    return {"ring": (ring, far, 0), "bridge": (bridge, [c(3, 0), c(6, 3), c(3, 6), c(0, 3), c(5, 6), c(1, 0), c(0, 1)], 0)}, fork


def test_havannah_ring_and_bridge_known_answers():
    """A ring (six stones around an empty cell, havannah.cc:394-409), a bridge (two corners) — decided on exactly the closing
    move, by the oracle and by the host-compiled rule core; and a ring closed by the SECOND player."""
    gs = "havannah(board_size=4)"
    lines, _ = _havannah_lines(4)
    for name, (mine, theirs, winner) in lines.items():
        for first in (0, 1):                                   # the winning line played by player 0, then by player 1
            og = OracleGame(gs)
            st = og.new_initial_state()
            emu = Emu(gs, 1)
            seq = []
            for k in range(len(mine)):
                if first == 0:
                    seq += [mine[k]] + ([theirs[k]] if k + 1 < len(mine) else [])
                else:
                    seq += [theirs[k], mine[k]]
            for i, a in enumerate(seq):
                assert not st.is_terminal(), (name, first, i)
                assert emu.status()[1][0] == 0
                st.apply_action(a)
                emu.apply([a])
            assert emu.errors() == 0
            assert st.is_terminal(), (name, first)
            want = [1.0, -1.0] if first == 0 else [-1.0, 1.0]
            assert st.returns() == want
            cur, term, rets = emu.status()
            assert term[0] == 1 and rets[0].tolist() == want, (name, first, rets)


import glob as _glob
import json as _json

_GOLD = sorted(_glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "playthroughs", "*.json")))


@pytest.mark.parametrize("path", _GOLD, ids=[os.path.basename(p)[:-5] for p in _GOLD])
def test_rule_core_replays_reference_playthrough(path):
    """The reference's golden traces replayed on the host build of the rule cores (the CPU twin of
    test_gpu_parity_games.py::test_device_replays_reference_playthrough): terminal flag, player to move, legal actions,
    returns with the sign of zero, every printed tensor."""
    gold = _json.load(open(path, encoding="utf-8"))
    try:
        emu = Emu(gold["game"], 1)
    except Exception as e:   # a trace of a configuration the packed layouts do not hold
        pytest.skip(str(e))
    hdr = gold["header"]
    assert emu.info.num_distinct_actions == int(hdr["NumDistinctActions"])
    assert emu.info.max_game_length == int(hdr["MaxGameLength"])
    for k, g in enumerate(gold["states"]):
        if g["detailed"]:
            cur, term, rets = emu.status()
            assert bool(term[0]) == g["is_terminal"]
            assert int(cur[0]) == g["current_player"]
            if "legal_actions" in g:
                assert emu.legal()[0] == g["legal_actions"]
            if "returns" in g:
                assert rets[0].tolist() == g["returns"]
                assert [bool(np.signbit(x)) for x in rets[0]] == [t.startswith("-") for t in g["returns_text"]]
            for name, vals in g["tensors"].items():
                p = int(name[name.index("(") + 1:name.index(")")])
                t = emu.tensor(p, 0 if name.startswith("Observation") else 1)[0]
                np.testing.assert_array_equal(t, np.array(vals, dtype=np.float32), err_msg=name)
        if k < len(gold["actions"]):
            emu.apply([gold["actions"][k]])
            assert emu.errors() == 0
    assert emu.status()[1][0] == 1

"""GPU parity: the device MCTS (one tree per thread) vs the oracle's restatement of algorithms/mcts.cc, both fed
the same Philox decisions: root child visit counts, total rewards (exact doubles), proven outcomes, BestChild and
the number of simulations run must be identical for every tree.  Plus the reference's own outcome-level MCTS tests
(algorithms/mcts_test.cc:109-155: the solver proves tic_tac_toe positions)."""
import math

import numpy as np
import pytest
import torch

import open_spiel_b200 as b2
from oracle_lib import OracleGame, oracle_mcts

pytestmark = pytest.mark.gpu


def make_roots(game_string, n, max_prefix, seed):
    """n lanes advanced by random legal plies (same actions on the device batch and on oracle states)."""
    rng = np.random.RandomState(seed)
    game, og = b2.load_game(game_string), OracleGame(game_string)
    batch = game.new_batch(n)
    states = [og.new_initial_state() for _ in range(n)]
    ks = rng.randint(0, max_prefix + 1, size=n)
    for t in range(max_prefix):
        acts = np.full(n, -1, dtype=np.int32)
        for i, st in enumerate(states):
            if t < ks[i] and not st.is_terminal():
                la = st.legal_actions()
                a = la[rng.randint(len(la))]
                nxt = st.clone()
                nxt.apply_action(a)
                if nxt.is_terminal():
                    continue                  # keep roots non-terminal
                states[i] = nxt
                acts[i] = a
        batch.apply_actions(torch.from_numpy(acts).to(batch._dev))
    batch.check_errors()
    return game, batch, states


CASES = [
    # game, trees, prefix plies, sims, n_rollouts, solve
    ("tic_tac_toe", 64, 4, 400, 1, True),
    ("tic_tac_toe", 32, 3, 150, 3, False),
    ("connect_four", 48, 12, 300, 1, True),
    ("connect_four(rows=4,columns=5,x_in_row=3)", 32, 6, 400, 2, True),
    ("breakthrough(rows=6,columns=6)", 24, 10, 150, 1, True),
    ("hex(board_size=5)", 32, 8, 200, 1, True),
    ("hex(board_size=4,swap=True)", 24, 2, 200, 1, True),
    ("go(board_size=5)", 32, 10, 150, 1, True),
    ("go(board_size=9)", 16, 30, 40, 1, True),
    ("go(board_size=3,komi=0.5)", 32, 4, 300, 1, True),
    # mid-game roots on tiny boards: positional superko decides most playouts and tree descents, so the root's hash history
    # must reach the search's work lanes (VERDICT r01: only the host-compiled kernel body covered these)
    ("go(board_size=2)", 48, 5, 120, 2, False),
    ("go(board_size=2)", 48, 12, 80, 1, True),
    ("go(board_size=3)", 48, 8, 150, 1, True),
    ("go(board_size=3)", 32, 14, 100, 4, False),
    # n_rollouts not a power of two: 24-byte nodes, the reference's double accumulator
    ("connect_four", 24, 6, 200, 5, True),
    # next-tier games: pass moves inside the tree (othello), the three-edge flood (y), 256-bit boards (mnk)
    ("othello", 32, 30, 150, 1, True),
    ("othello", 24, 56, 300, 1, True),
    ("havannah(board_size=3)", 32, 4, 300, 1, True),
    ("havannah(board_size=4,swap=True)", 24, 10, 150, 1, True),
    ("y(board_size=5)", 32, 4, 300, 1, True),
    ("y(board_size=9)", 24, 12, 120, 2, False),
    ("mnk(m=5,n=5,k=4)", 32, 6, 200, 1, True),
    ("mnk", 8, 10, 60, 1, True),
]

# node budget + garbage collection (MCTSBot max_memory_mb -> max_nodes_, mcts.cc:205-231, 441-482): game, trees, prefix, sims,
# n_rollouts, solve, budget (max_nodes_ per tree)
GC_CASES = [
    ("connect_four", 32, 6, 3000, 1, False, 300),
    ("tic_tac_toe", 32, 2, 1500, 2, True, 120),
    ("hex(board_size=4)", 24, 2, 2500, 1, True, 400),
    ("go(board_size=5)", 16, 6, 1200, 1, True, 600),
    ("breakthrough(rows=5,columns=4)", 16, 3, 1500, 1, False, 250),
    ("go(board_size=9)", 8, 20, 600, 1, True, 3000),
    ("othello", 16, 10, 1200, 1, False, 300),
    ("mnk(m=4,n=4,k=3)", 16, 2, 1500, 2, True, 350),
]


PUCT_CASES = [
    ("tic_tac_toe", 48, 4, 300, 1, True),
    ("connect_four", 32, 10, 300, 1, True),
    ("breakthrough(rows=6,columns=6)", 16, 8, 150, 1, False),
    ("go(board_size=5)", 24, 8, 150, 1, True),
]


@pytest.mark.parametrize("gs,n,prefix,sims,nroll,solve", CASES, ids=["%s-%d" % (c[0], c[3]) for c in CASES])
def test_device_mcts_equals_oracle_mcts(gs, n, prefix, sims, nroll, solve):
    _check_against_oracle(gs, n, prefix, sims, nroll, solve, puct=False)


@pytest.mark.parametrize("gs,n,prefix,sims,nroll,solve", PUCT_CASES, ids=["%s-%d" % (c[0], c[3]) for c in PUCT_CASES])
def test_device_puct_equals_oracle_puct(gs, n, prefix, sims, nroll, solve):
    """ChildSelectionPolicy::PUCT (mcts.cc:103-112, 328-335) with the rollout evaluator's uniform prior."""
    _check_against_oracle(gs, n, prefix, sims, nroll, solve, puct=True)


@pytest.mark.parametrize("gs,n,prefix,sims,nroll,solve,budget", GC_CASES, ids=["%s-%d" % (c[0], c[3]) for c in GC_CASES])
def test_device_garbage_collection_equals_oracle(gs, n, prefix, sims, nroll, solve, budget):
    """The oracle's collector is pinned to the unmodified reference bit for bit (tests/test_mcts_oracle_vs_reference.py);
    the device must collect after the same simulations and end with identical root statistics."""
    collections = _check_against_oracle(gs, n, prefix, sims, nroll, solve, puct=False, budget=budget)
    assert collections >= n


def test_wall_clock_budget_stops_the_search():
    """max_wall_clock_time (mcts.cc:362-365): simulations stop once the budget has passed; everything run so far is kept."""
    game = b2.load_game("go(board_size=9)")
    batch = game.new_batch(256)
    out = b2.mcts_search(batch, 1000000, seed=3, max_wall_clock_time=0.25, max_nodes_total=256 * 200000)
    ran = out["sims_run"].cpu().numpy()
    assert (ran > 0).all() and (ran < 1000000).all()
    assert bool((out["visits"].sum(dim=1).cpu().numpy() == ran - 1).all())
    assert batch.error_count()[0] == 0


def _check_against_oracle(gs, n, prefix, sims, nroll, solve, puct, budget=0):
    game, batch, states = make_roots(gs, n, prefix, seed=sum(map(ord, gs)) % 1000)
    seed, offset = 0xC0FFEE, 17
    out = b2.mcts_search(batch, sims, uct_c=2.0, n_rollouts=nroll, solve=solve, seed=seed, tree_index_offset=offset,
                         child_selection_policy=b2.ChildSelectionPolicy.PUCT if puct else b2.ChildSelectionPolicy.UCT,
                         max_nodes_per_tree=budget)
    assert batch.error_count()[0] == 0
    visits, reward = out["visits"].cpu().numpy(), out["total_reward"].cpu().numpy()
    outcome, best, ran = out["outcome_p0"].cpu().numpy(), out["best_action"].cpu().numpy(), out["sims_run"].cpu().numpy()
    gcs = out["gc_runs"].cpu().numpy()
    collections = 0
    for i, st in enumerate(states):
        o = oracle_mcts(st, 2.0, sims, nroll, solve, seed, tree_index=i + offset, puct=puct, max_nodes=budget or 1)
        assert ran[i] == o["sims_run"], (gs, i)
        assert gcs[i] == o["gc_runs"], (gs, i)
        collections += o["gc_runs"]
        assert int(visits[i].sum()) == sum(v for _, v, _, _ in o["children"])
        for a, v, r, oc in o["children"]:
            assert visits[i, a] == v, (gs, i, a)
            assert reward[i, a] == r, (gs, i, a, reward[i, a], r)            # exact double equality
            assert (math.isnan(oc) and math.isnan(outcome[i, a])) or outcome[i, a] == oc, (gs, i, a)
        illegal = sorted(set(range(game.num_distinct_actions())) - {a for a, _, _, _ in o["children"]})
        assert not visits[i, illegal].any()
        assert best[i] == o["best_action"], (gs, i)
    return collections


def _solve(game_string, actions, sims=10000):
    """GetOutcome-style helper of mcts_test.cc:100-107: search from the position after `actions`."""
    game = b2.load_game(game_string)
    st = game.new_initial_state()
    for a in actions:
        st.apply_action(a)
    bot = b2.MCTSBot(game, b2.RandomRolloutEvaluator(20, 42), 2.0, sims, solve=True, seed=42)
    out = bot.mcts_search(st)
    legal = st.legal_actions()
    return st, out, legal


def test_solver_proves_tic_tac_toe_positions():
    # mcts_test.cc:123-134 MCTSTest_SolveDraw: "x(1,1) o(0,0) x(2,2)" -> o to move, proven draw, best move o(2,0) or o(0,2)
    st, out, legal = _solve("tic_tac_toe", [4, 0, 8])
    oc = out["outcome_p0"][0].cpu().numpy()
    assert st.current_player() == 1 and int(out["sims_run"].item()) < 10000       # root proven -> early exit
    assert not np.isnan(oc[legal]).any() and (oc[legal] >= 0).all()               # no winning move for o
    assert int(out["best_action"].item()) in (6, 2) and oc[int(out["best_action"].item())] == 0
    # mcts_test.cc:136-143 SolveLoss: "x(1,1) o(0,0) x(2,2) o(0,1) x(0,2)" -> every o move is a proven loss
    st, out, legal = _solve("tic_tac_toe", [4, 0, 8, 1, 2])
    oc = out["outcome_p0"][0].cpu().numpy()
    assert st.current_player() == 1 and (oc[legal] == 1).all()
    # mcts_test.cc:145-152 SolveWin: "x(0,1) o(2,2)" -> x wins with x(0,2)
    st, out, legal = _solve("tic_tac_toe", [1, 8])
    assert st.current_player() == 0
    assert int(out["best_action"].item()) == 2 and float(out["outcome_p0"][0, 2].item()) == 1.0
    assert int(out["sims_run"].item()) < 10000


def test_mcts_root_invariants_many_trees():
    """Deterministic facts of algorithms/mcts.cc that hold for every tree: sum of child visits = sims - 1 when the
    root is unproven (the first simulation stops at the root), children = LegalActions, runs are reproducible."""
    game = b2.load_game("connect_four")
    n, sims = 4096, 64
    batch = game.new_batch(n)
    out = b2.mcts_search(batch, sims, solve=False, seed=5)
    v = out["visits"]
    assert bool((v.sum(dim=1) == sims - 1).all())
    assert bool((out["sims_run"] == sims).all())
    out2 = b2.mcts_search(batch, sims, solve=False, seed=5)
    assert torch.equal(out["visits"], out2["visits"]) and torch.equal(out["total_reward"], out2["total_reward"])
    out3 = b2.mcts_search(batch, sims, solve=False, seed=6)
    assert not torch.equal(out["visits"], out3["visits"])
    # different trees use different random streams
    assert len({tuple(r) for r in v[:64].cpu().tolist()}) > 32


def test_device_mcts_matches_reference_mctsbot_in_distribution():
    """The reference's RNG streams (std::shuffle, absl::Uniform) cannot be reproduced (SURVEY §8c), so against the
    UNMODIFIED MCTSBot the comparison is statistical: over many independent searches of the same connect_four
    position, the mean share of simulations each root action receives must agree (uct_c = 2, 400 simulations, no
    solver), and so must the mean root value.  The reference's means are stored (tests/reference_golden.py)."""
    from reference_golden import expected
    gs, prefix = "connect_four", [3, 3, 2]
    sims, trees = 400, 512
    game = b2.load_game(gs)
    batch = game.new_batch(trees)
    for a in prefix:
        batch.apply_actions(torch.full((trees,), a, dtype=torch.int32, device=batch._dev))
    out = b2.mcts_search(batch, sims, uct_c=2.0, n_rollouts=1, solve=False, seed=2024)
    v = out["visits"].double()
    dev_share = (v / v.sum(dim=1, keepdim=True)).mean(dim=0).cpu().numpy()
    dev_value = float((out["total_reward"].sum(dim=1) / v.sum(dim=1)).mean())
    ref = expected("gpu_mcts/connect_four")
    share, value = np.array(ref["share"]), ref["value"]
    # standard error of a mean share over a few hundred searches is ~0.005; allow 0.03
    assert np.abs(dev_share - share).max() < 0.03, (dev_share, share)
    assert abs(dev_value - value) < 0.05, (dev_value, value)


def reference_golden():
    """The unmodified MCTSBot's mean root shares and value over 256 searches (seeds 1..256) of the position above."""
    import ref_lib
    rg = ref_lib.RefGame("connect_four")
    st = rg.new_initial_state()
    for a in [3, 3, 2]:
        st.apply_action(a)
    n_ref = 256
    share = np.zeros(7)
    value = 0.0
    for seed in range(n_ref):
        r = ref_lib.ref_mcts(rg, st, 2.0, 400, 1, False, seed + 1)
        tot = sum(vv for _, vv, _ in r["children"])
        for a, vv, _ in r["children"]:
            share[a] += vv / tot / n_ref
        value += sum(rw for _, _, rw in r["children"]) / tot / n_ref
    return {"gpu_mcts/connect_four": {"share": share.tolist(), "value": value}}

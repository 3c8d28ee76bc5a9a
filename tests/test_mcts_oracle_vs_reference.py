"""CPU: pins the oracle's MCTS (oracle/algorithms/mcts.cc) to the UNMODIFIED reference's MCTSBot (algorithms/mcts.cc, built by
oracle/ref_build.mk).  Fed the reference's own random streams — std::mt19937(seed) for the bot (std::shuffle of new
children) and for the RandomRolloutEvaluator (absl::Uniform over the legal actions) — the restatement must reproduce the
search BIT FOR BIT: the root's children in the same (shuffled) order, their visit counts, their total rewards as exact
doubles, and BestChild.  The device kernel is then compared with the same oracle code on the Philox stream
(tests/test_gpu_mcts.py): the two modes differ only in where the random integers come from.  The reference's searches are
stored (tests/reference_golden.py)."""
import random

import pytest

from oracle_lib import OracleGame, oracle_mcts
from reference_golden import expected

CASES = [
    # game, prefix plies, simulations, n_rollouts, solve, seed
    ("tic_tac_toe", 0, 500, 1, True, 1),
    ("tic_tac_toe", 3, 300, 4, True, 7),
    ("tic_tac_toe", 2, 400, 1, False, 3),
    ("connect_four", 0, 600, 1, True, 42),
    ("connect_four", 9, 400, 2, True, 5),
    ("breakthrough(rows=6,columns=6)", 4, 200, 1, True, 11),
    ("hex(board_size=5)", 3, 300, 1, True, 2),
    ("go(board_size=5)", 6, 150, 1, True, 9),
    ("go(board_size=9)", 10, 60, 1, True, 13),
    # next-tier games: the oracle's rule restatements under the unmodified MCTSBot's search, bit for bit
    ("othello", 20, 150, 1, True, 21),
    ("othello", 54, 400, 1, True, 22),
    ("mnk(m=5,n=5,k=4)", 6, 200, 1, True, 23),
    ("y(board_size=5)", 4, 300, 1, True, 24),
    ("havannah(board_size=3)", 4, 300, 1, True, 25),
    ("havannah(board_size=4,swap=True)", 10, 150, 2, True, 26),
]


GC_CASES = [("connect_four", 12000, 3), ("hex(board_size=4)", 9000, 5)]


def start(game, gs, prefix, seed):
    rng = random.Random(seed)
    s = game.new_initial_state()
    for _ in range(prefix):
        a = rng.choice(s.legal_actions())
        nxt = s.clone()
        nxt.apply_action(a)
        if nxt.is_terminal():
            break
        s.apply_action(a)
    return s


def reference_golden():
    import ref_lib
    out = {}
    for gs, prefix, sims, nroll, solve, seed in CASES:
        rg = ref_lib.RefGame(gs)
        out["mcts/%s-%d" % (gs, sims)] = ref_lib.ref_mcts(rg, start(rg, gs, prefix, seed), 2.0, sims, nroll, solve, seed)
    for gs, sims, seed in GC_CASES:
        rg = ref_lib.RefGame(gs)
        r = ref_lib.ref_mcts(rg, rg.new_initial_state(), 2.0, sims, 1, False, seed, max_memory_mb=1)
        out["mcts_gc/%s" % gs] = dict(r, sizeof_search_node=ref_lib.sizeof_search_node())
    return out


@pytest.mark.parametrize("gs,prefix,sims,nroll,solve,seed", CASES, ids=["%s-%d" % (c[0], c[2]) for c in CASES])
def test_oracle_mcts_equals_reference_mctsbot_bitwise(gs, prefix, sims, nroll, solve, seed):
    ref = expected("mcts/%s-%d" % (gs, sims))
    mine = oracle_mcts(start(OracleGame(gs), gs, prefix, seed), 2.0, sims, nroll, solve, seed, reference_rng=True)
    assert [c[0] for c in mine["children"]] == [c[0] for c in ref["children"]]          # same shuffled child order
    assert [c[1] for c in mine["children"]] == [c[1] for c in ref["children"]]          # visit counts
    assert [c[2] for c in mine["children"]] == [c[2] for c in ref["children"]]          # total rewards, exact doubles
    assert mine["best_action"] == ref["best_action"]
    assert mine["root_visits"] == ref["root_visits"]


@pytest.mark.parametrize("gs,sims,seed", GC_CASES)
def test_oracle_garbage_collection_equals_reference_bitwise(gs, sims, seed):
    """MCTSBot's node budget (max_memory_mb -> max_nodes_, mcts.cc:205-231) and GarbageCollect (mcts.cc:441-482): with
    max_memory_mb = 1 the tree is collected several times inside these searches; the oracle must prune the same nodes at
    the same simulations (same gc_limit_ trajectory), i.e. reproduce the final root statistics bit for bit."""
    ref = expected("mcts_gc/%s" % gs)
    os_ = OracleGame(gs).new_initial_state()
    max_nodes = (1 << 20) // ref["sizeof_search_node"] + 1
    mine = oracle_mcts(os_, 2.0, sims, 1, False, seed, reference_rng=True, max_nodes=max_nodes)
    assert mine["gc_runs"] >= 2, mine["gc_runs"]
    assert mine["children"] and [list(c[:3]) for c in mine["children"]] == ref["children"]
    assert mine["best_action"] == ref["best_action"] and mine["root_visits"] == ref["root_visits"]
    # and the budget changes the search: without it the statistics differ
    free = oracle_mcts(os_, 2.0, sims, 1, False, seed, reference_rng=True)
    assert free["gc_runs"] == 0 and [c[:3] for c in free["children"]] != [c[:3] for c in mine["children"]]

"""CPU: pins the oracle's external-sampling MCCFR (oracle/algorithms/mccfr.cc) to the UNMODIFIED reference's
ExternalSamplingMCCFRSolver (algorithms/external_sampling_mccfr.cc, built by oracle/ref_build.mk).  Fed the reference's own
random stream (std::mt19937 + std::uniform_real_distribution, both libstdc++), one traversal per update, the restatement
must reproduce the reference's tables BIT FOR BIT — same information states visited, same cumulative regrets, same
cumulative policy.  The reference's tables are stored as digests (tests/reference_golden.py)."""
import pytest

from oracle_lib import OracleGame, OracleMCCFR
from reference_golden import digest, expected

CASES = [("kuhn_poker", 0, [1, 9, 90, 900]), ("kuhn_poker", 12345, [50, 500]), ("leduc_poker", 0, [1, 20, 400]), ("leduc_poker", 7, [1000])]


def table_digest(t):
    return digest({k: [v["legal"], v["regrets"], v["cum_policy"]] for k, v in t.items()})


def checkpoints(solver, steps):
    out = []
    for k in steps:
        solver.iterate(k)
        out.append(table_digest(solver.table()))
    return out


def reference_golden():
    import ref_lib
    out = {"mccfr/%s-%d" % (name, seed): checkpoints(ref_lib.RefMCCFR(ref_lib.RefGame(name), seed), steps)
           for name, seed, steps in CASES}
    ref = ref_lib.RefMCCFR(ref_lib.RefGame("kuhn_poker"), 39823987)
    ref.iterate(1000)
    out["mccfr/known_answer/kuhn_poker"] = {"nash_conv": ref.nash_conv(), "table": table_digest(ref.table())}
    return out


@pytest.mark.parametrize("name,seed,steps", CASES)
def test_oracle_mccfr_equals_reference_bitwise(name, seed, steps):
    mine = OracleMCCFR(OracleGame(name), seed=seed, rng_mode=0, traversals_per_update=1)
    assert checkpoints(mine, steps) == expected("mccfr/%s-%d" % (name, seed))


def test_reference_known_answer_kuhn_nash_conv():
    """external_sampling_mccfr_test.cc: 1000 iterations on kuhn_poker reach NashConv < 0.05 (loose bound of the reference
    test); the restatement with the same stream has the same tables, so the same NashConv."""
    want = expected("mccfr/known_answer/kuhn_poker")
    assert want["nash_conv"] < 0.1
    mine = OracleMCCFR(OracleGame("kuhn_poker"), seed=39823987, rng_mode=0, traversals_per_update=1)
    mine.iterate(1000)
    assert table_digest(mine.table()) == want["table"]


def test_position_keyed_stream_batches_are_order_independent():
    """Philox mode: K traversals per update read frozen tables, so running them is deterministic and K = 1 differs from
    K = 8 only by the documented semantics (sanity: both converge on kuhn)."""
    a = OracleMCCFR(OracleGame("kuhn_poker"), seed=5, rng_mode=1, traversals_per_update=8)
    b = OracleMCCFR(OracleGame("kuhn_poker"), seed=5, rng_mode=1, traversals_per_update=8)
    a.iterate(40)
    b.iterate(40)
    assert a.table() == b.table()

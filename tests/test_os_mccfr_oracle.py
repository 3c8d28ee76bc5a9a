"""CPU: pins the oracle's outcome-sampling MCCFR (oracle/algorithms/os_mccfr.cc) and the kFull averaging of its
external-sampling MCCFR to the UNMODIFIED reference solvers (algorithms/outcome_sampling_mccfr.cc,
external_sampling_mccfr.cc:188-230, built by oracle/ref_build.mk).  Fed the reference's own random stream — std::mt19937
through the uniform_real / discrete distributions of the abseil shim the reference is built against — with one episode per
update, the restatements must reproduce the reference's tables BIT FOR BIT.  The reference's tables are stored as digests (tests/reference_golden.py)."""
import pytest

from oracle_lib import OracleGame, OracleMCCFR, OracleOSMCCFR
from reference_golden import expected
from test_mccfr_oracle import checkpoints, table_digest

OS_CASES = [("kuhn_poker", 0, 0.6, [1, 9, 90, 900]), ("kuhn_poker", 1234, 0.3, [50, 2000]), ("leduc_poker", 0, 0.6, [1, 20, 400, 3000]),
            ("leduc_poker", 7, 0.9, [1500])]
FULL_CASES = [("kuhn_poker", 3, [1, 30, 300]), ("leduc_poker", 5, [1, 10, 60])]


def reference_golden():
    import ref_lib
    out = {}
    for name, seed, eps, steps in OS_CASES:
        out["os_mccfr/%s-%d" % (name, seed)] = checkpoints(ref_lib.RefOSMCCFR(ref_lib.RefGame(name), seed, eps), steps)
    for name, seed, steps in FULL_CASES:
        out["mccfr_full/%s-%d" % (name, seed)] = checkpoints(ref_lib.RefMCCFR(ref_lib.RefGame(name), seed, full_average=True), steps)
    ref = ref_lib.RefOSMCCFR(ref_lib.RefGame("kuhn_poker"), 39823987)
    ref.iterate(10000)
    out["os_mccfr/known_answer/kuhn_poker"] = {"nash_conv": ref.nash_conv(), "table": table_digest(ref.table())}
    return out


@pytest.mark.parametrize("name,seed,eps,steps", OS_CASES)
def test_oracle_outcome_sampling_equals_reference_bitwise(name, seed, eps, steps):
    mine = OracleOSMCCFR(OracleGame(name), seed=seed, rng_mode=0, trajectories_per_update=1, epsilon=eps)
    assert checkpoints(mine, steps) == expected("os_mccfr/%s-%d" % (name, seed))


@pytest.mark.parametrize("name,seed,steps", FULL_CASES)
def test_oracle_full_average_equals_reference_bitwise(name, seed, steps):
    mine = OracleMCCFR(OracleGame(name), seed=seed, rng_mode=0, traversals_per_update=1, full_average=True)
    assert checkpoints(mine, steps) == expected("mccfr_full/%s-%d" % (name, seed))


def test_reference_known_answer_outcome_sampling_kuhn():
    """outcome_sampling_mccfr_test.cc: 10000 iterations on kuhn_poker give NashConv < 0.17 with its seed; the restatement
    with the same stream reaches the same tables."""
    want = expected("os_mccfr/known_answer/kuhn_poker")
    assert want["nash_conv"] < 0.17
    mine = OracleOSMCCFR(OracleGame("kuhn_poker"), seed=39823987, rng_mode=0, trajectories_per_update=1)
    mine.iterate(10000)
    assert table_digest(mine.table()) == want["table"]

"""CPU: pins the oracle's CFR restatement against the UNMODIFIED reference CFRSolver: identical tables, bit for bit,
after every one of several iterations on kuhn_poker and leduc_poker — the reference's own "two implementations agree"
criterion (python/algorithms/cfr_test.py:240-272), tightened from 1e-10 to exact — plus the known answers of
algorithms/cfr_test.cc (Kuhn exploitability, Leduc NashConv).  The reference's side is stored (tests/reference_golden.py)."""
import pytest

from oracle_lib import OracleCFR, OracleGame
from reference_golden import digest, expected

CASES = [("kuhn_poker", [1, 1, 3, 5, 40]), ("leduc_poker", [1, 1, 3])]
FIELDS = ("legal", "regrets", "cum_policy", "cur_policy")


def table_digest(t):
    return digest({k: [v[f] for f in FIELDS] for k, v in t.items()})


def checkpoints(solver, iters):
    out = []
    for k in iters:
        solver.iterate(k)
        out.append([len(solver.table()), table_digest(solver.table())])
    return out


def reference_golden():
    import ref_lib
    out = {"cfr/%s" % gs: checkpoints(ref_lib.RefCFR(ref_lib.RefGame(gs)), iters) for gs, iters in CASES}
    # cfr_test.cc:36-62 — Kuhn: exploitability <= 0.05 after 300 iterations; cfr_test.cc:299-301 Leduc NashConv <= 2 after 10
    r = ref_lib.RefCFR(ref_lib.RefGame("kuhn_poker"))
    r.iterate(300)
    out["cfr/known_answer/kuhn_poker"] = {"exploitability": r.exploitability(), "table": table_digest(r.table())}
    r = ref_lib.RefCFR(ref_lib.RefGame("leduc_poker"))
    r.iterate(10)
    out["cfr/known_answer/leduc_poker"] = {"nash_conv": r.nash_conv(), "table": table_digest(r.table())}
    return out


@pytest.mark.parametrize("gs,iters", CASES)
def test_oracle_cfr_tables_equal_reference_bitwise(gs, iters):
    want = expected("cfr/" + gs)
    for k, (mine, ref) in enumerate(zip(checkpoints(OracleCFR(OracleGame(gs)), iters), want)):
        assert ref[0] == {"kuhn_poker": 12, "leduc_poker": 936}[gs]
        assert mine == ref, (gs, "checkpoint", k)


def test_reference_known_answers():
    # the reference's values, and the oracle reaches the same tables, hence the same values
    kuhn, leduc = expected("cfr/known_answer/kuhn_poker"), expected("cfr/known_answer/leduc_poker")
    assert kuhn["exploitability"] <= 0.05
    assert leduc["nash_conv"] <= 2.0
    for gs, iters, want in (("kuhn_poker", 300, kuhn), ("leduc_poker", 10, leduc)):
        o = OracleCFR(OracleGame(gs))
        o.iterate(iters)
        assert table_digest(o.table()) == want["table"], gs


def test_oracle_cfr_converges_on_kuhn():
    # average policy at "0" (player 0 holding the jack): never... sanity on known Kuhn structure:
    o = OracleCFR(OracleGame("kuhn_poker"))
    o.iterate(300)
    t = o.table()
    assert len(t) == 12
    # with the king facing a bet ("2pb"), calling is dominant: average policy puts ~all mass on bet/call
    cp = t["2pb"]["cum_policy"]
    assert cp[1] / (cp[0] + cp[1]) > 0.99
    # with the jack facing a bet ("0pb"), folding is dominant
    cp = t["0pb"]["cum_policy"]
    assert cp[0] / (cp[0] + cp[1]) > 0.99

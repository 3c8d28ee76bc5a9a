"""GPU parity: device-resident CFR vs the oracle's restatement of algorithms/cfr.cc and vs the unmodified reference (its
tables and NashConv values stored, tests/reference_golden.py): cumulative regrets, cumulative policy and current policy of every
information state, BIT FOR BIT (north-star tolerance is 1e-6), after several iteration counts; tree sizes and
information-state counts of integration_tests/api_test.py:77-104."""
import numpy as np
import pytest

import open_spiel_b200 as b2
from oracle_lib import OracleCFR, OracleGame, infostate_tensors
from reference_golden import expected
from test_cfr_oracle import table_digest

pytestmark = pytest.mark.gpu

TOL = 1e-6      # north-star tolerance; the assertions below demand exact equality and report the max |delta|


def compare(dev_table, cpu_table, tensors):
    by_key = {dev_table["keys"][k].tobytes(): k for k in range(len(dev_table["players"]))}
    assert len(by_key) == len(cpu_table)
    worst = 0.0
    for key, v in cpu_table.items():
        k = by_key[tensors[key]]
        lo, hi = dev_table["offsets"][k], dev_table["offsets"][k + 1]
        assert dev_table["legal_actions"][lo:hi].tolist() == v["legal"]
        for f in ("regrets", "cum_policy", "cur_policy"):
            d = dev_table[f][lo:hi]
            c = np.array(v[f])
            worst = max(worst, float(np.abs(d - c).max()))
            assert np.array_equal(d, c), (key, f, d, c)
    assert worst <= TOL
    return worst


@pytest.mark.parametrize("gs,steps,plus", [("kuhn_poker", [1, 1, 3, 45, 250], False), ("leduc_poker", [1, 1, 2, 6], False),
                                           ("kuhn_poker", [1, 2, 47], True), ("leduc_poker", [1, 3], True)])
def test_device_cfr_equals_oracle_bitwise(gs, steps, plus):
    game, og = b2.load_game(gs), OracleGame(gs)
    dev = b2.CFRSolver(game, linear_averaging=plus, regret_matching_plus=plus)
    cpu = OracleCFR(og, linear_averaging=plus, regret_matching_plus=plus)
    tensors = infostate_tensors(og)
    info = dev.info()
    expect = {"kuhn_poker": (4, 24, 30, 12), "leduc_poker": (157, 3780, 5520, 936)}[gs]   # api_test.py:77-104
    assert (info.chance_nodes, info.decision_nodes, info.terminal_nodes, info.num_infosets) == expect
    for k in steps:
        dev.evaluate_and_update_policy(k)
        cpu.iterate(k)
        compare(dev.table(), cpu.table(), tensors)


REF_CASES = [("kuhn_poker", 300), ("leduc_poker", 25)]
NASH_CONV_CASES = [("kuhn_poker", [1, 10, 100, 300]), ("leduc_poker", [1, 5, 20])]


def as_reference_table(dev_table, tensors):
    """The device table keyed by information-state string, shaped like the reference's CFRSolver table."""
    by_key = {dev_table["keys"][k].tobytes(): k for k in range(len(dev_table["players"]))}
    assert len(by_key) == len(tensors)
    out = {}
    for key, blob in tensors.items():
        k = by_key[blob]
        lo, hi = dev_table["offsets"][k], dev_table["offsets"][k + 1]
        out[key] = {"legal": dev_table["legal_actions"][lo:hi].tolist(),
                    **{f: dev_table[f][lo:hi].tolist() for f in ("regrets", "cum_policy", "cur_policy")}}
    return out


def reference_golden():
    import ref_lib
    out = {}
    for gs, iters in REF_CASES:
        ref = ref_lib.RefCFR(ref_lib.RefGame(gs))
        ref.iterate(iters)
        out["gpu_cfr/%s-%d" % (gs, iters)] = {"table": table_digest(ref.table()), "exploitability": ref.exploitability()}
    for gs, checkpoints in NASH_CONV_CASES:
        ref = ref_lib.RefCFR(ref_lib.RefGame(gs))
        done, vals = 0, []
        for it in checkpoints:
            ref.iterate(it - done)
            done = it
            vals.append([ref.nash_conv(), ref.exploitability()])
        out["gpu_cfr/nash_conv/" + gs] = vals
    return out


@pytest.mark.parametrize("gs,iters", REF_CASES)
def test_device_cfr_equals_unmodified_reference(gs, iters):
    want = expected("gpu_cfr/%s-%d" % (gs, iters))
    game = b2.load_game(gs)
    dev = b2.CFRSolver(game)
    dev.evaluate_and_update_policy(iters)
    tensors = infostate_tensors(OracleGame(gs))
    assert table_digest(as_reference_table(dev.table(), tensors)) == want["table"]
    if gs == "kuhn_poker":
        assert want["exploitability"] <= 0.05          # cfr_test.cc:36-62, now also true of the device tables


def test_checkpoint_resume_is_exact():
    game = b2.load_game("kuhn_poker")
    a, b = b2.CFRSolver(game), b2.CFRSolver(game)
    a.evaluate_and_update_policy(20)
    t = a.table()
    b.load_table(t["regrets"], t["cum_policy"], t["cur_policy"], iteration=20)
    a.evaluate_and_update_policy(15)
    b.evaluate_and_update_policy(15)
    ta, tb = a.table(), b.table()
    for f in ("regrets", "cum_policy", "cur_policy"):
        assert np.array_equal(ta[f], tb[f])


def test_sharded_traversal_path_is_bit_identical():
    """The multi-GPU code path (traverse_shard -> all-reduce -> apply_deltas) run on one GPU: with 1 shard, and with 3 and
    8 shards evaluated one after the other and their contribution buffers summed by hand (what the NCCL all-reduce does:
    every slot is one rank's value plus zeros).  Tables must equal the single-GPU kernel's bit for bit — the summation
    order problem of a per-entry partial-sum exchange (SURVEY §7 "CFR floating point") does not arise."""
    import torch
    from open_spiel_b200 import parallel
    from open_spiel_b200._lib import check, lib
    for plus in (False, True):
        game = b2.load_game("leduc_poker")
        ref = b2.CFRSolver(game, linear_averaging=plus, regret_matching_plus=plus)
        ref.evaluate_and_update_policy(60)
        tr = ref.table()
        one = parallel.DistributedCFRSolver(game, linear_averaging=plus, regret_matching_plus=plus, in_library=False)
        one.evaluate_and_update_policy(60)
        tables = [one.table()]
        for shards in (3, 8):
            multi = parallel.DistributedCFRSolver(game, linear_averaging=plus, regret_matching_plus=plus, in_library=False)
            L, h = lib(), multi.solver._h
            for it in range(1, 61):
                for player in (0, 1):
                    acc = torch.zeros_like(multi.delta)
                    for shard in range(shards):
                        check(L.b2s_cfr_traverse_shard(h, player, it, shard, shards, None))
                        torch.cuda.synchronize()
                        acc += multi.delta
                    multi.delta.copy_(acc)
                    check(L.b2s_cfr_apply_deltas(h, None))
            tables.append(multi.table())
        for t in tables:
            for f in ("regrets", "cum_policy", "cur_policy"):
                assert np.array_equal(t[f], tr[f]), (plus, f)
        assert np.abs(tr["regrets"]).max() > 0.1       # the tables are not trivially zero


@pytest.mark.parametrize("gs,checkpoints", NASH_CONV_CASES)
def test_device_nash_conv_matches_reference(gs, checkpoints):
    """The evaluation step of the CFR loop (examples/cfr_example.cc:37-46): NashConv / Exploitability of the average
    policy, device vs the unmodified reference's tabular_exploitability.cc, to 1e-9."""
    game = b2.load_game(gs)
    dev = b2.CFRSolver(game)
    done = 0
    for it, (ref_nash_conv, ref_exploitability) in zip(checkpoints, expected("gpu_cfr/nash_conv/" + gs)):
        dev.evaluate_and_update_policy(it - done)
        done = it
        assert abs(dev.nash_conv() - ref_nash_conv) <= 1e-9, (gs, it)
        assert abs(dev.exploitability() - ref_exploitability) <= 1e-9
    if gs == "kuhn_poker":
        assert dev.exploitability() <= 0.05                      # cfr_test.cc:36-62
        assert abs(dev.last_values[2] - (-1.0 / 18.0)) <= 1e-3   # game value for player 0 (cfr_test.cc:40-41)
    else:
        assert dev.nash_conv() <= 2.0                            # cfr_test.cc:299-301 (after >= 10 iterations)


@pytest.mark.parametrize("gs,iters", [("kuhn_poker", 40), ("leduc_poker", 25)])
def test_best_response_actions_achieve_the_best_response_values(gs, iters):
    """b2s_cfr_best_response (TabularBestResponse::GetBestResponseActions, best_response.cc:194-228): for each player, the pure
    policy made of the reported actions, played against the other player's average policy, earns exactly the best-response
    value that NashConv is built from — checked on the device by evaluating that profile as a current policy."""
    game = b2.load_game(gs)
    s = b2.CFRSolver(game)
    s.evaluate_and_update_policy(iters)
    actions, vals = s.best_response(average=True)
    nc = s.nash_conv(average=True)
    assert nc == pytest.approx((vals[0] - vals[2]) + (vals[1] - vals[3]), abs=1e-15)
    t = s.table()
    off, players, legal = t["offsets"], t["players"], t["legal_actions"]
    avg = np.empty_like(t["cum_policy"])
    for i in range(len(players)):
        lo, hi = off[i], off[i + 1]
        tot = t["cum_policy"][lo:hi].sum()
        avg[lo:hi] = t["cum_policy"][lo:hi] / tot if tot > 0 else 1.0 / (hi - lo)
    for b in (0, 1):
        prof = avg.copy()
        for i in range(len(players)):
            if players[i] == b:
                lo, hi = off[i], off[i + 1]
                assert actions[i] in legal[lo:hi]
                prof[lo:hi] = (legal[lo:hi] == actions[i]).astype(np.float64)
        probe = b2.CFRSolver(game)
        probe.load_table(cur_policy=prof)
        probe.nash_conv(average=False)
        on_policy_value_of_b = probe.last_values[2 + b]
        assert on_policy_value_of_b == pytest.approx(vals[b], abs=1e-12), (gs, b)
        assert vals[b] >= vals[2 + b] - 1e-12                     # a best response is at least as good as the policy itself

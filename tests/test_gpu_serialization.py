"""GPU: training state crosses the boundary in the reference's own text format, in both directions, without losing a bit:
device CFR tables -> CFRSolverBase::Serialize text -> the UNMODIFIED reference's DeserializeCFRSolver -> both continue
training -> tables still identical; and reference text -> device solver.  Plus State::Serialize round trips.  The
reference's side is stored (tests/reference_golden.py): digests of its texts and tables, its state texts and strings."""
import numpy as np
import pytest

import open_spiel_b200 as b2
from oracle_lib import OracleGame, infostate_tensors
from reference_golden import digest, expected
from test_gpu_cfr import as_reference_table

pytestmark = pytest.mark.gpu

TABLE_CASES = [("kuhn_poker", 25), ("leduc_poker", 7)]
STATE_GAMES = ("connect_four", "go(board_size=5)", "leduc_poker", "othello", "havannah(board_size=4,swap=True)", "y(board_size=5)",
               "mnk(m=4,n=4,k=3)")


def entries_digest(text):
    """The set of table entries of a serialized solver (the reference emits its unordered_map in hash order)."""
    parts = text.partition("[SolverValuesTable]\n")[2].split("<~>")
    return digest(sorted(zip(parts[0::2], parts[1::2])))


def table_digest(t):
    return digest({k: [v["regrets"], v["cum_policy"], v["cur_policy"]] for k, v in t.items()})


def infostate_events(st, rng, pick):
    """Information-state strings and chance outcomes along one random playout (actions drawn by `pick`)."""
    out = []
    while not st.is_terminal():
        if st.current_player() >= 0:
            out.append(st.information_state_string(st.current_player()))
        else:
            out.append([[a for a, _ in st.chance_outcomes()], [p for _, p in st.chance_outcomes()]])
        la = st.legal_actions()
        a = int(la[rng.randint(len(la))])
        pick(a)
        st.apply_action(a)
    return out


def average_policy_digest(pol):
    return digest({k: [[a for a, _ in v], [p for _, p in v]] for k, v in pol.items()})


def reference_golden():
    import ref_lib
    from test_serialization import _layout_from
    from open_spiel_b200 import serialization as ser
    out = {}
    for name, iters in TABLE_CASES:
        rg = ref_lib.RefGame(name)
        ref = ref_lib.RefCFR(rg)
        ref.iterate(iters)
        keys, layout = _layout_from(ref.table(), name)
        text = ser.serialize_cfr_solver(ref_lib.game_to_string(rg), "CFRSolver", iters, keys, layout)
        e = {"text": entries_digest(ref_lib.cfr_serialize(ref))}
        ref = ref_lib.cfr_deserialize(rg, text)                 # stock DeserializeCFRSolver on the text we write
        e["loaded"] = table_digest(ref.table())
        ref.iterate(4)
        e["plus_4"] = table_digest(ref.table())
        e["text_plus_4"] = entries_digest(ref_lib.cfr_serialize(ref))
        ref.iterate(3)
        e["plus_7"] = table_digest(ref.table())
        out["gpu_serialization/cfr/" + name] = e
    rng = np.random.RandomState(5)
    for gs in STATE_GAMES:
        rg = ref_lib.RefGame(gs)
        st = rg.new_initial_state()
        for _ in range(9):
            if st.is_terminal():
                break
            la = st.legal_actions()
            st.apply_action(int(la[rng.randint(len(la))]))
        text = ref_lib.state_serialize(st)
        rs = ref_lib.deserialize_state(rg, text)
        out["gpu_serialization/state/" + gs] = {"text": text, "history": rs.history(), "legal": rs.legal_actions()}
    rng = np.random.RandomState(11)
    for name in ("kuhn_poker", "leduc_poker"):
        rg = ref_lib.RefGame(name)
        events = [infostate_events(rg.new_initial_state(), rng, lambda a: None) for _ in range(6)]
        ref = ref_lib.RefCFR(rg)
        ref.iterate(9)
        pol = {}
        for key, v in ref.table().items():
            total = 0.0
            for c in v["cum_policy"]:          # sequential sum as CFRAveragePolicy does (Python 3.12's sum() is compensated)
                total += c
            pol[key] = list(zip(v["legal"], [c / total if total > 0 else 1.0 / len(v["legal"]) for c in v["cum_policy"]]))
        out["gpu_serialization/infostate/" + name] = {"events": events, "average_policy": average_policy_digest(pol)}
    return out


@pytest.mark.parametrize("name,iters", TABLE_CASES)
def test_device_tables_to_reference_and_back(name, iters):
    want = expected("gpu_serialization/cfr/" + name)
    game = b2.load_game(name)
    tensors = infostate_tensors(OracleGame(name))
    dev = b2.CFRSolver(game)
    dev.evaluate_and_update_policy(iters)
    text = dev.serialize()
    assert entries_digest(text) == want["text"]             # the reference's own text, up to the order of entries
    assert table_digest(as_reference_table(dev.table(), tensors)) == want["loaded"]   # what stock DeserializeCFRSolver loads
    dev.evaluate_and_update_policy(4)
    assert table_digest(as_reference_table(dev.table(), tensors)) == want["plus_4"]   # the reference continued from it exactly
    # and the other way: a fresh device solver resumes from the reference's text (ours, which equals it up to entry order)
    text = dev.serialize()
    assert entries_digest(text) == want["text_plus_4"]
    dev2 = b2.CFRSolver(game)
    parsed = dev2.load_serialized(text)
    assert parsed["iteration"] == iters + 4 and dev2.info().iteration == iters + 4
    dev2.evaluate_and_update_policy(3)
    assert table_digest(as_reference_table(dev2.table(), tensors)) == want["plus_7"]


def test_state_serialize_round_trip_through_the_reference():
    rng = np.random.RandomState(5)
    for gs in STATE_GAMES:
        want = expected("gpu_serialization/state/" + gs)
        game = b2.load_game(gs)
        st = game.new_initial_state()
        for _ in range(9):
            if st.is_terminal():
                break
            la = st.legal_actions()
            st.apply_action(int(la[rng.randint(len(la))]))
        text = st.serialize()
        assert text == want["text"]                         # the reference's State::Serialize of the same state
        assert want["history"] == st.history() and want["legal"] == st.legal_actions()   # the reference loads it so
        back = game.deserialize_state(want["text"])         # and we load the reference's
        assert back.history() == st.history() and back.legal_actions() == st.legal_actions()
        assert np.array_equal(np.asarray(back.observation_tensor(0)), np.asarray(st.observation_tensor(0)))


def test_information_state_strings_and_tabular_policy_match_the_reference():
    rng = np.random.RandomState(11)
    for name in ("kuhn_poker", "leduc_poker"):
        want = expected("gpu_serialization/infostate/" + name)
        game = b2.load_game(name)
        for ref_events in want["events"]:
            assert infostate_events(game.new_initial_state(), rng, lambda a: None) == ref_events
        dev = b2.CFRSolver(game)
        dev.evaluate_and_update_policy(9)
        # the reference's CFRAveragePolicy of its own tables after 9 iterations
        assert average_policy_digest(dev.tabular_average_policy()) == want["average_policy"]

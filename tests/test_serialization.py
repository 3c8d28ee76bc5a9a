"""CPU: the text formats of open_spiel_b200/serialization.py against the UNMODIFIED reference: information-state strings
rebuilt from tensors, hex-float doubles, CFRSolverBase::Serialize / DeserializeCFRSolver in both directions (the reference
loads what we write; we parse what it writes), State::Serialize.  The reference's side is stored (tests/reference_golden.py);
the CFR tables behind it come from the oracle's CFRSolver, which reproduces the reference's bit for bit
(test_cfr_oracle.py)."""
import ctypes
import random
import struct

import numpy as np
import pytest

from open_spiel_b200 import serialization as ser
from oracle_lib import OracleCFR, OracleGame, infostate_tensors
from reference_golden import digest, expected


def test_hex_double_is_printf_percent_a():
    libc = ctypes.CDLL(None)
    libc.snprintf.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_double]

    def c_a(x):
        b = ctypes.create_string_buffer(64)
        libc.snprintf(b, 64, b"%a", ctypes.c_double(x))
        return b.value.decode()

    rnd = random.Random(7)
    vals = [0.0, -0.0, 1.0, -1.0, 0.5, 1e-6, 1 / 3, 5e-324, 2.2250738585072014e-308, 1.7976931348623157e308, 0.1]
    vals += [struct.unpack("<d", struct.pack("<Q", rnd.getrandbits(64)))[0] for _ in range(20000)]
    for v in vals:
        if v == v:
            assert ser.hex_double(v) == c_a(v)
            assert ser.parse_double(ser.hex_double(v)) == v or v in (float("inf"), float("-inf"))


@pytest.mark.parametrize("name", ["kuhn_poker", "leduc_poker"])
def test_information_state_strings_from_tensors(name):
    # every information state of the game: the oracle's string (pinned to the reference playthroughs) vs ours from its tensor
    tensors = infostate_tensors(OracleGame(name))
    assert len(tensors) == {"kuhn_poker": 12, "leduc_poker": 936}[name]
    f = ser.INFORMATION_STATE_STRING[name]
    for key, blob in tensors.items():
        assert f(np.frombuffer(blob, dtype=np.float32)) == key


def _layout_from(ref_table, name):
    """A CFRSolver.table()-shaped dict (flat arrays + offsets + tensor keys) holding the reference's table."""
    tensors = infostate_tensors(OracleGame(name))
    keys = sorted(ref_table)
    offsets, legal = [0], []
    cols = {f: [] for f in ("regrets", "cum_policy", "cur_policy")}
    for k in keys:
        v = ref_table[k]
        legal += v["legal"]
        for f in cols:
            cols[f] += v[f]
        offsets.append(len(legal))
    t = {"offsets": np.array(offsets, dtype=np.int32), "legal_actions": np.array(legal, dtype=np.int32),
         "keys": np.stack([np.frombuffer(tensors[k], dtype=np.float32) for k in keys])}
    t.update({f: np.array(v) for f, v in cols.items()})
    return keys, t


CFR_CASES = [("kuhn_poker", 37), ("leduc_poker", 6)]
STATE_GAMES = ["connect_four", "go(board_size=5)", "kuhn_poker", "leduc_poker", "breakthrough"]


def entries_digest(text):
    """The header of a serialized solver and the set of its table entries (the reference emits its unordered_map in hash
    order, so only the order of entries may differ)."""
    head, _, vals = text.partition("[SolverValuesTable]\n")
    parts = vals.split(ser.DELIMITER)
    return digest(head, sorted(zip(parts[0::2], parts[1::2])))


def table_digest(t):
    return digest({k: [v["legal"], v["regrets"], v["cum_policy"], v["cur_policy"]] for k, v in t.items()})


def random_history(game, rng, plies=12):
    st = game.new_initial_state()
    hist = []
    for _ in range(plies):
        if st.is_terminal():
            break
        a = rng.choice(st.legal_actions())
        st.apply_action(a)
        hist.append(a)
    return st, hist


def reference_golden():
    import ref_lib
    out = {}
    for name, iters in CFR_CASES:
        rg = ref_lib.RefGame(name)
        ref = ref_lib.RefCFR(rg)
        ref.iterate(iters)
        text = ref_lib.cfr_serialize(ref)
        keys, layout = _layout_from(ref.table(), name)
        mine = ser.serialize_cfr_solver(ref_lib.game_to_string(rg), "CFRSolver", iters, keys, layout)
        loaded = ref_lib.cfr_deserialize(rg, mine)           # the reference loads what we write ...
        first = table_digest(loaded.table())
        loaded.iterate(3)                                     # ... and continues training from it
        out["serialization/cfr/" + name] = {"game": ref_lib.game_to_string(rg), "text": entries_digest(text),
                                            "parsed": table_digest(ser.deserialize_cfr_solver(text)["table"]),
                                            "loaded": first, "loaded_plus_3": table_digest(loaded.table())}
    for gs in STATE_GAMES:
        rg = ref_lib.RefGame(gs)
        st, hist = random_history(rg, random.Random(3))
        text = ref_lib.state_serialize(st)
        back = ref_lib.deserialize_state(rg, text)
        out["serialization/state/" + gs] = {"text": text, "history": back.history(), "to_string": back.to_string()}
    return out


@pytest.mark.parametrize("name,iters", CFR_CASES)
def test_cfr_solver_text_format_both_directions(name, iters):
    want = expected("serialization/cfr/" + name)
    o = OracleCFR(OracleGame(name))              # the reference's CFRSolver tables, bit for bit (test_cfr_oracle.py)
    o.iterate(iters)
    table = o.table()
    # (1) we write what the reference writes: same header, same set of table entries byte for byte
    keys, layout = _layout_from(table, name)
    assert ser.table_keys(name, layout) == keys
    mine = ser.serialize_cfr_solver(want["game"], "CFRSolver", iters, keys, layout)
    assert entries_digest(mine) == want["text"]
    # (2) so we parse what the reference writes: its text is ours up to the order of entries
    parsed = ser.deserialize_cfr_solver(mine)
    assert parsed["game"] == want["game"] and parsed["solver_type"] == "CFRSolver" and parsed["iteration"] == iters
    assert table_digest(parsed["table"]) == want["parsed"] == table_digest(table)
    # (3) the reference loads what we write, and continues training from it exactly like the original
    assert want["loaded"] == table_digest(table)
    o.iterate(3)
    assert want["loaded_plus_3"] == table_digest(o.table())
    # (4) and back into flat arrays in a given row order (CFRSolver.load_table's arguments)
    r, c, p = ser.table_arrays_from(parsed["table"], keys, layout)
    assert np.array_equal(r, layout["regrets"]) and np.array_equal(c, layout["cum_policy"]) and np.array_equal(p, layout["cur_policy"])


@pytest.mark.parametrize("gs", STATE_GAMES)
def test_state_serialize_format(gs):
    want = expected("serialization/state/" + gs)
    st, hist = random_history(OracleGame(gs), random.Random(3))
    text = ser.serialize_state(hist)
    assert text == want["text"]
    # the reference's state deserialized from that text
    assert want["history"] == hist and want["to_string"] == st.to_string()

"""Pins oracle/policy.c: generated label lists == the frozen lists of engine/tests/legacyconstants.h:162,2438,4757
and generated FLAT_PLANE_IDX == policymaprepresentation.h:39,2314,4633 (element by element against the tables recorded
in tests/golden/policy_tables_reference.json, and through SHA-256 + spot values in tests/golden/policy_tables.json)."""
import ctypes
import hashlib
import json
import os

import pytest

from oracle.chess import Position, lib

GOLD = os.path.join(os.path.dirname(__file__), "golden", "policy_tables.json")
MODES = {"crazyhouse": 0, "chess": 1, "lichess": 2}


def _tables(mode):
    L = lib()
    L.opolicy_label.restype = ctypes.c_char_p
    n = L.opolicy_nb_labels(mode)
    return [L.opolicy_label(mode, i).decode() for i in range(n)], [L.opolicy_flat_plane_idx(mode, i) for i in range(n)]


@pytest.mark.parametrize("name", sorted(MODES))
def test_tables_match_golden_hashes(name):
    g = json.load(open(GOLD))[name]
    labels, flat = _tables(MODES[name])
    assert len(labels) == g["n"]
    assert hashlib.sha256(",".join(labels).encode()).hexdigest() == g["labels_sha256"]
    assert hashlib.sha256(",".join(map(str, flat)).encode()).hexdigest() == g["flat_sha256"]
    for lab, (idx, fl) in g["spot"].items():
        assert labels[idx] == lab and flat[idx] == fl


def test_tables_match_reference_sources():
    """Element by element against the tables of the reference's sources (tests/golden/policy_tables_reference.json,
    recorded by gen_policy_tables_golden.py)."""
    ref = json.load(open(os.path.join(os.path.dirname(GOLD), "policy_tables_reference.json")))
    for name in ("crazyhouse", "lichess", "chess"):
        labels, flat = _tables(MODES[name])
        assert flat == ref[name]["flat_plane_idx"], name
        assert labels == ref[name]["labels"].split(","), name


def test_move_index_semantics():
    L = lib()
    L.opolicy_move_index.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_int, ctypes.c_int]
    # white e2e4: queen-move plane N, length 2 -> channel 1, origin e2 (=12)
    p = Position(variant="crazyhouse")
    assert L.opolicy_move_index(p._buf, p.move_from_uci("e2e4"), 0, 1) == 1 * 64 + 12
    # black reply e7e5 is mirrored to e2e4 (node.cpp:970-977)
    p.push_uci("e2e4")
    assert L.opolicy_move_index(p._buf, p.move_from_uci("e7e5"), 0, 1) == 1 * 64 + 12
    # classic (non policy-map) index = label index of the (mirrored) UCI string
    labels, _ = _tables(0)
    assert L.opolicy_move_index(p._buf, p.move_from_uci("g8f6"), 0, 0) == labels.index("g1f3")
    # castling: classical chess uses e1g1, chess960 king-takes-rook (sfutil.cpp:199-285)
    c = Position("r3k2r/8/8/8/8/8/8/R3K2R w KQkq - 0 1")
    labels_c, flat_c = _tables(1)
    assert L.opolicy_move_index(c._buf, c.move_from_uci("e1g1"), 1, 0) == labels_c.index("e1g1")
    c960 = Position("r3k2r/8/8/8/8/8/8/R3K2R w HAha - 0 1", "chess", True)
    assert L.opolicy_move_index(c960._buf, c960.move_from_uci("e1h1"), 1, 0) == labels_c.index("e1h1")
    # every legal move of a few positions has a label, and indices are unique per position
    for fen, var in ((None, "crazyhouse"), ("5r2/ppp2pkp/3p4/2bP4/2Pnp1N1/3P2pP/PP2n1P1/R2Q1R1K[PBRQnbb] w - - 0 28", "crazyhouse"),
                     ("1k1r3r/pppb1p2/2nbqn1p/3p2p1/3PP1P1/3Q1PP1/PPN2NBP/R1B2RK1[p] b - - 0 12", "crazyhouse")):
        q = Position(fen, var)
        idx = [L.opolicy_move_index(q._buf, m, 0, 1) for m in q.legal_moves()]
        assert min(idx) >= 0 and len(set(idx)) == len(idx)

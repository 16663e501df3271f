"""ThreadManager's stop / prolong rules (manager/threadmanager.cpp:114-178) as the C-ABI's pure functions.
The expected verdicts are worked out by hand from the reference's formulas."""
from crazyara_b200.engine import TimeControl, continue_search, early_stopping


def _tc(**kw):
    base = dict(movetime_ms=1000.0, update_interval_ms=250.0, overall_nps=10000.0, safe_remaining_ms=60000.0,
                move_overhead_ms=20.0, last_value_eval=0.1, in_game=1, can_prolong=1)
    base.update(kw)
    return TimeControl(**base)


def test_early_stopping_is_off_outside_games_and_without_nps():
    args = (500.0, 10 ** 6, 1, 900, 10, 0.5, 0.1)
    assert early_stopping(_tc(), *args) == 1
    assert early_stopping(_tc(in_game=0), *args) == 0
    assert early_stopping(_tc(overall_nps=0.0), *args) == 0


def test_max_nodes_rule():
    # node count above 2 x NPS x move time (20000) and the most visited child also has the best Q
    tc = _tc()
    assert early_stopping(tc, 750.0, 20001, 1, 100, 90, 0.0, 0.5) == 1
    assert early_stopping(tc, 750.0, 20000, 1, 100, 90, 0.0, 0.5) == 0      # not strictly above
    assert early_stopping(tc, 750.0, 20001, 0, 100, 90, 0.0, 0.5) == 0      # best Q elsewhere


def test_second_move_cannot_catch_up_rule():
    tc = _tc()
    # remaining 250 ms x 10 nodes/ms = 2500 more visits: 1000 + 2500 < 2 x 1800 and Q(first) > Q(second)
    assert early_stopping(tc, 250.0, 5000, 0, 1800, 1000, 0.3, 0.2) == 2
    assert early_stopping(tc, 250.0, 5000, 0, 1750, 1000, 0.3, 0.2) == 0    # 3500 < 3500 fails
    assert early_stopping(tc, 250.0, 5000, 0, 1800, 1000, 0.2, 0.3) == 0    # the runner-up has the better Q
    assert early_stopping(tc, 500.0, 5000, 0, 1800, 1000, 0.3, 0.2) == 0    # too much time left


def test_continue_search_rules():
    tc = _tc()
    # the evaluation dropped below the last move's: prolong once, remember the new evaluation
    assert continue_search(tc, 500.0, -0.2, 0, 0.1) == (True, 1, -0.20000000298023224)
    assert continue_search(tc, 500.0, -0.3, 1, -0.2)[0:2] == (True, 2)
    assert continue_search(tc, 500.0, -0.4, 2, -0.3)[0] is False             # at most twice
    assert continue_search(tc, 500.0, 0.2, 0, 0.1) == (False, 0, 0.10000000149011612)  # no drop
    assert continue_search(tc, 269.0, -0.2, 0, 0.1)[0] is False              # less than interval + overhead left
    assert continue_search(_tc(can_prolong=0), 500.0, -0.2, 0, 0.1)[0] is False
    assert continue_search(_tc(in_game=0), 500.0, -0.2, 0, 0.1)[0] is False
    assert continue_search(_tc(overall_nps=0.0), 500.0, -0.2, 0, 0.1)[0] is False
    assert continue_search(_tc(safe_remaining_ms=1999.0), 500.0, -0.2, 0, 0.1)[0] is False  # 2 x move time would flag


def test_root_statistics_match_the_oracle_tree():
    """collect_time_stats (device code, 1-lane host emulation) against the same quantities read off the oracle's root."""
    import numpy as np
    from oracle import search as osr
    from oracle.chess import Position
    from tests.hostemu import HeSearch, HeState
    for variant, vid, mode, moves, sims in (("chess", 0, "chess", ["d2d4", "d7d5"], 800),
                                            ("crazyhouse", 1, "crazyhouse", ["e2e4"], 500),
                                            ("chess", 0, "chess", [], 60)):
        st = osr.default_settings(mode, batch_size=16, simulations=sims, node_policy_temperature=1.0)
        pos = Position(None, variant, False)
        pos.push_uci(*moves)
        he = HeState(Position(None, variant, False).fen(), vid, False)
        for m in moves:
            he.do_move(he.move_from_uci(m))
        S, H = osr.Search(st), HeSearch(st)
        ro = S.run(pos, osr.fake_net(S.n_labels), with_keys=True)
        H.run(he, osr.fake_net(H.n_labels), with_keys=True)
        ts = H.time_stats()
        visits, q = ro["visits"].astype(np.int64), ro["q"]
        # first_and_second_max (util/blazeutil.h:154-178): strict comparisons, first maximum wins
        a1 = int(np.argmax(visits))
        rest = visits.copy()
        rest[a1] = -1
        a2 = int(np.argmax(rest)) if len(visits) > 1 and rest.max() > 0 else 0
        assert ts["valid"] == 1 and ts["node_count"] == ro["nodes"] and ro["free_visits"] == 0
        assert ts["first_visits"] == visits[a1] and ts["second_visits"] == (visits[a2] if a2 != a1 or len(visits) == 1 else 0)
        assert ts["q_first"] == q[a1] and ts["q_second"] == q[a2]
        assert ts["max_q_is_max_visits"] == int(int(np.argmax(q)) == a1)
        assert ts["value_eval"] == q[a1]                       # updated_value_eval of an unsolved root


def test_first_and_second_max_reference_vectors():
    """The reference's own known-answer test of first_and_second_max (tests.cpp:626-646), through the device code that
    applies it to the root's visit counts (collect_time_stats); the Q values tell which children were picked."""
    import ctypes
    import numpy as np
    from tests.hostemu import lib
    L = lib()
    L.he_time_stats_of.argtypes = [ctypes.c_int] + [ctypes.c_void_p] * 4

    def stats(visits):
        n = np.array(visits, np.uint32)
        q = (np.arange(len(visits)) * 0.01 - 0.5).astype(np.float32)      # q[i] identifies child i
        i, f = np.zeros(3, np.uint32), np.zeros(3, np.float32)
        L.he_time_stats_of(len(visits), n.ctypes.data, q.ctypes.data, i.ctypes.data, f.ctypes.data)
        return int(i[0]), int(i[1]), int(round((f[0] + 0.5) * 100)), int(round((f[1] + 0.5) * 100)), float(f[2]), q

    first, second, a1, a2, eval_, q = stats([3, 42, 1, 3, 99, 8, 7])
    assert (first, second, a1, a2) == (99, 42, 4, 1) and eval_ == q[4]
    first, second, a1, a2, eval_, q = stats([99, 3, 1, 3, 42, 8, 7])
    assert (first, second, a1, a2) == (99, 42, 0, 4) and eval_ == q[0]
    # ties: the first maximum wins both ranks (strict comparisons)
    assert stats([5, 5, 5])[:4] == (5, 5, 0, 1)
    assert stats([7])[:4] == (7, 0, 0, 0)


def _ara_time_for_move(row):
    import ctypes
    from crazyara_b200 import lib
    L = lib()
    L.ara_time_for_move.argtypes = [ctypes.c_long] + [ctypes.c_int] * 5
    movetime, wtime, btime, winc, binc, movestogo, overhead, me, move_number = row[:9]
    return L.ara_time_for_move(movetime, (wtime, btime)[me], (winc, binc)[me], movestogo, overhead, move_number)


def test_time_for_move_equals_the_reference_golden():
    """ara_time_for_move against outputs of the UNMODIFIED reference TimeManager (tests/golden/timeman.json, generated
    by tests/golden/gen_timeman_golden.py from oracle/_ref)."""
    import json
    import os
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "timeman.json")))
    assert len(g["rows"]) > 2000
    bad = [r for r in g["rows"] if _ara_time_for_move(r) != r[9]]
    assert bad == []


def test_time_for_move_equals_the_compiled_reference_live():
    """The same on 5000 seeded random inputs, against what the compiled reference (oracle/_ref/libref_parts.so) returned
    for them (tests/golden/timeman_random.json, recorded by tests/golden/gen_timeman_golden.py)."""
    import json
    import os
    from tests.golden.gen_timeman_golden import random_rows
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "timeman_random.json")))
    rows = random_rows()
    assert len(rows) == len(g["reference_ms"]) == 5000
    for row, ref_ms in zip(rows, g["reference_ms"]):
        assert _ara_time_for_move(row) == ref_ms, row

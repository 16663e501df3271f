"""Generates tests/golden/timeman.json from the UNMODIFIED reference TimeManager (oracle/_ref/libref_parts.so, built by
`make -C oracle ref` from /root/reference/engine/src/manager/timemanager.cpp + agents/config/searchlimits.cpp).
Run in the build container (the GPU box has no /root/reference):  python tests/golden/gen_timeman_golden.py"""
import ctypes
import itertools
import json
import os
import random

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))


def cases():
    yield from ((mt, 0, 0, 0, 0, 0, ov, me, 1) for mt, ov, me in itertools.product((1, 15, 40, 220, 5000), (0, 20, 50), (0, 1)))
    clock = itertools.product((500, 1999, 20000, 60000, 600000, 7200000), (0, 100, 101, 2000, 12345), (0, 1, 5, 40),
                              (0, 20, 100), (1, 12, 34, 35, 36, 80))
    for i, (t, inc, mtg, ov, mn) in enumerate(clock):
        me = i & 1
        yield (0, t if me == 0 else 7, 7 if me == 0 else t, inc if me == 0 else 3, 3 if me == 0 else inc, mtg, ov, me, mn)
    yield (0, 0, 0, 0, 0, 0, 20, 0, 1)      # nothing given: 1000 ms less the overhead
    yield (0, 0, 0, 0, 0, 30, 20, 1, 5)     # movestogo without a clock


def random_rows(n=5000, seed=11):
    """Random (movetime, wtime, btime, winc, binc, movestogo, move_overhead, me, move_number) rows, 80 % with a clock."""
    rng = random.Random(seed)
    rows = []
    for _ in range(n):
        clock = rng.random() < 0.8
        rows.append((0 if clock else rng.choice((0, 1, 30, 250, 4000)), rng.randrange(0, 3000000) if clock else 0,
                     rng.randrange(0, 3000000) if clock else 0, rng.randrange(0, 30000), rng.randrange(0, 30000),
                     rng.choice((0, 0, 0, 1, 7, 40)), rng.choice((0, 20, 100, 500)), rng.randrange(2), rng.randrange(1, 120)))
    return rows


def main():
    L = ctypes.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_parts.so"))
    L.ref_time_for_move.argtypes = [ctypes.c_long] + [ctypes.c_int] * 8
    rows = [list(c) + [L.ref_time_for_move(*c)] for c in cases()]
    json.dump({"columns": ["movetime", "wtime", "btime", "winc", "binc", "movestogo", "move_overhead", "me", "move_number",
                           "reference_ms"], "rows": rows}, open(os.path.join(HERE, "timeman.json"), "w"), separators=(",", ":"))
    json.dump({"reference_ms": [L.ref_time_for_move(*r) for r in random_rows()]},
              open(os.path.join(HERE, "timeman_random.json"), "w"), separators=(",", ":"))
    print(len(rows), "cases")


if __name__ == "__main__":
    main()

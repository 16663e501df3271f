"""Generates tests/golden/ref_misc.json from the UNMODIFIED reference PGN writer and chess960 generator
(oracle/_ref/libref_parts.so, `make -C oracle ref`).  Run in the build container:
    python tests/golden/gen_ref_misc_golden.py"""
import ctypes
import json
import os
import random

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))

PGN_CASES = [
    dict(header=["standard", "SelfPlay", "2026.01.01 12:00:00", "Darmstadt, GER", "?",
                 "rnbqkbnr/pppppppp/8/8/8/8/PPPPPPPP/RNBQKBNR w KQkq - 0 1", "A", "B", "0-1", "?"],
         moves=["f3", "e5", "g4", "Qh4#"]),
    dict(header=["crazyhouse", "SelfPlay", "d", "s", "?", "fen", "w", "b", "?", "?"], moves=[]),
    dict(header=["chess960", "SelfPlay", "d", "s", "3", "fen", "w", "b", "1/2-1/2", "40/9000"], moves=["a"] * 8),
    dict(header=["3check", "E", "d", "s", "?", "fen", "w", "b", "1-0", "?"],
         moves=["e4", "e5", "Nf3", "Nc6", "Bb5", "a6", "Ba4", "Nf6", "O-O", "Be7", "Re1", "b5", "Bb3", "d6", "c3", "O-O",
                "h3"]),
]


def random_pgn_cases():
    """Seeded games of 0 to 120 moves drawn from SAN spellings that exercise castling, promotions, drops and checks."""
    rng = random.Random(5)
    cases = []
    for n in (0, 1, 2, 7, 8, 9, 16, 33, 120):
        moves = [rng.choice(["e4", "Nf3", "O-O", "exd5", "Q@h5+", "a8Q", "Rad1", "N@f7#"]) for _ in range(n)]
        header = ["crazyhouse960", "SelfPlay", "2026.09.24 10:00:00", "Darmstadt, GER", "?", "some fen", "x", "y",
                  rng.choice(["1-0", "0-1", "1/2-1/2"]), "?"]
        cases.append(dict(header=header, moves=moves))
    return cases


def render(L, case):
    hdr = (ctypes.c_char_p * 10)(*[h.encode() for h in case["header"]])
    n = len(case["moves"])
    mv = (ctypes.c_char_p * max(n, 1))(*[m.encode() for m in case["moves"]] or [b""])
    out = ctypes.create_string_buffer(1 << 16)
    assert L.ref_pgn_render(hdr, mv, n, out, 1 << 16) >= 0
    return out.value.decode()


def main():
    L = ctypes.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_parts.so"))
    buf = ctypes.create_string_buffer(128)
    fens = set()
    for seed in range(30000):
        L.ref_chess960_fen(seed, buf)
        fens.add(buf.value.decode())
    ranks = sorted(f.split("/")[7].split(" ")[0] for f in fens)
    tails = sorted({f.split("/", 1)[1].split("/", 6)[0] + "|" + f.split(" ", 1)[1] for f in fens})
    json.dump({"pgn": [dict(c, text=render(L, c)) for c in PGN_CASES], "chess960_back_ranks": ranks,
               "chess960_fen_shape": tails}, open(os.path.join(HERE, "ref_misc.json"), "w"), separators=(",", ":"))
    json.dump({"text": [render(L, c) for c in random_pgn_cases()]}, open(os.path.join(HERE, "ref_pgn_random.json"), "w"),
              separators=(",", ":"))
    print(len(ranks), "distinct chess960 set-ups,", len(PGN_CASES), "pgn cases")


if __name__ == "__main__":
    main()

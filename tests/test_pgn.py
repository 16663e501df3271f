"""SAN spelling and PGN layout of the reference (environments/chess_related/board.cpp:277-385, rl/gamepgn.cpp:27-55).
Host-side code only (the state functions of the C-ABI do no GPU work)."""
import pytest

from crazyara_b200.engine import BoardState
from crazyara_b200.pgn import GamePGN, result_string
from crazyara_b200.export import BLACK_WIN, DRAWN, WHITE_WIN


def _san(fen, uci, variant=0, is960=False, win=False):
    return BoardState().set(fen, is960, variant).action_to_san(uci, win)


def test_reference_ambiguity_case():
    # tests.cpp:184-200: Nf3-d2 with the other knight on b3 -> ambiguous by rank only, so the FILE names the origin
    assert _san("r1bq1rk1/ppppbppp/2n2n2/4p3/4P3/1N1P1N2/PPP2PPP/R1BQKB1R w KQ - 5 6", "f3d2") == "Nfd2"


@pytest.mark.parametrize("fen,uci,variant,san", [
    ("rnbqkbnr/pppppppp/8/8/8/8/PPPPPPPP/RNBQKBNR w KQkq - 0 1", "e2e4", 0, "e4"),
    ("rnbqkbnr/pppppppp/8/8/8/8/PPPPPPPP/RNBQKBNR w KQkq - 0 1", "g1f3", 0, "Nf3"),
    ("rnbqkbnr/ppp1pppp/8/3p4/4P3/8/PPPP1PPP/RNBQKBNR w KQkq d6 0 2", "e4d5", 0, "exd5"),
    ("rnbqkbnr/ppp1p1pp/8/3pPp2/8/8/PPPP1PPP/RNBQKBNR w KQkq f6 0 3", "e5f6", 0, "exf6"),            # en passant
    ("r3k2r/8/8/8/8/8/8/R3K2R w KQkq - 0 1", "e1g1", 0, "O-O"),
    ("r3k2r/8/8/8/8/8/8/R3K2R b KQkq - 0 1", "e8c8", 0, "O-O-O"),
    ("7k/P7/8/8/8/8/8/K7 w - - 0 1", "a7a8q", 0, "a8Q+"),                                              # no '='
    ("1n5k/P7/8/8/8/8/8/K7 w - - 0 1", "a7b8n", 0, "axb8N"),
    ("7k/8/R7/8/8/8/R7/4K3 w - - 0 1", "a2a4", 0, "R2a4"),                                            # same file -> rank
    ("8/7k/8/Q7/8/8/8/Q1Q1K3 w - - 0 1", "a1c3", 0, "Qa1c3"),                                          # file and rank taken
    ("6k1/5ppp/8/8/8/8/8/R3K3 w - - 0 1", "a1a8", 0, "Ra8+"),
    ("rnbqkbnr/pppppppp/8/8/8/8/PPPPPPPP/RNBQKBNR[Nq] w KQkq - 0 1", "N@f3", 1, "N@f3"),             # crazyhouse drop
    ("rnbqkbnr/pppp1ppp/8/4p3/8/8/PPPPPPPP/RNBQKBNR[Q] w KQkq - 0 2", "Q@h5", 1, "Q@h5"),
])
def test_san_spelling(fen, uci, variant, san):
    assert _san(fen, uci, variant) == san


def test_chess960_castling_is_spelled_by_side():
    # king b1, rooks a1 / g1: the move is "king takes rook" (b1g1 / b1a1) in the 960 encoding
    fen = "1k6/8/8/8/8/8/8/RK4R1 w KQ - 0 1"
    st = BoardState().set(fen, True, 0)
    sans = {st.action_to_uci(a): st.action_to_san(a) for a in st.legal_actions()}
    assert sans["b1g1"] == "O-O" and sans["b1a1"] == "O-O-O"


def test_every_legal_move_has_a_distinct_san():
    for fen, v in (("r1bq1rk1/ppppbppp/2n2n2/4p3/4P3/1N1P1N2/PPP2PPP/R1BQKB1R w KQ - 5 6", 0),
                   ("r2q1rk1/ppp2ppp/2np1n2/2b1p1B1/2B1P1b1/2NP1N2/PPP2PPP/R2Q1RK1[Pn] w - - 0 8", 1)):
        st = BoardState().set(fen, False, v)
        sans = [st.action_to_san(a) for a in st.legal_actions()]
        assert len(set(sans)) == len(sans)


def test_game_pgn_layout_and_mate_marker(tmp_path):
    g = GamePGN("chess", False, "A", "B", date="2026.01.01 12:00:00")
    st = BoardState().set("", False, 0)
    g.fen = st.fen()
    for u in ("f2f3", "e7e5", "g2g4"):
        assert g.play_move(st, u) == 4
    assert g.play_move(st, "d8h4") == 0          # fool's mate: the side to move has lost
    g.result = result_string(BLACK_WIN)
    text = str(g)
    assert text == ('[Variant "standard"]\n[Event "SelfPlay"]\n[Date "2026.01.01 12:00:00"]\n[Site "Darmstadt, GER"]\n'
                    '[Round "?"]\n[FEN "rnbqkbnr/pppppppp/8/8/8/8/PPPPPPPP/RNBQKBNR w KQkq - 0 1"]\n[White "A"]\n'
                    '[Black "B"]\n[Result "0-1"]\n[PlyCount "4"]\n[TimeControl "?"]\n\n'
                    '1. f3 e5 2. g4 Qh4# 0-1\n\n')
    path = str(tmp_path / "games.pgn")
    g.write(path)
    g.write(path)
    assert open(path).read() == (text + "\n") * 2
    assert GamePGN("crazyhouse", True).variant == "crazyhouse960" and GamePGN(0, True).variant == "chess960"
    assert [result_string(r) for r in (WHITE_WIN, BLACK_WIN, DRAWN)] == ["1-0", "0-1", "1/2-1/2"]


def test_line_break_every_eight_plies():
    g = GamePGN("chess", date="d")
    g.game_moves = ["a"] * 9
    assert str(g).split("\n\n", 1)[1] == "1. a a 2. a a 3. a a 4. a a \n5. a ?\n\n"


def _game_from(case):
    g = GamePGN("chess", date=case["header"][2])
    (g.variant, g.event, g.date, g.site, g.round, g.fen, g.white, g.black, g.result, g.time_control) = case["header"]
    g.game_moves = list(case["moves"])
    return g


def test_pgn_text_equals_the_reference_writer_golden():
    """str(GamePGN) against the text the UNMODIFIED reference `operator<<(ostream&, GamePGN)` wrote for the same record
    (tests/golden/ref_misc.json, generated from oracle/_ref by tests/golden/gen_ref_misc_golden.py)."""
    import json
    import os
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "ref_misc.json")))
    assert len(g["pgn"]) >= 4
    for case in g["pgn"]:
        assert str(_game_from(case)) == case["text"]


def test_pgn_text_equals_the_compiled_reference_live():
    """Seeded random games (0 to 120 moves) against the text the compiled reference writer produced for them
    (tests/golden/ref_pgn_random.json, recorded by tests/golden/gen_ref_misc_golden.py)."""
    import json
    import os
    from tests.golden.gen_ref_misc_golden import random_pgn_cases
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "ref_pgn_random.json")))
    cases = random_pgn_cases()
    assert len(cases) == len(g["text"]) == 9
    for case, text in zip(cases, g["text"]):
        assert str(_game_from(case)) == text

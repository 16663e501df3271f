"""Training-sample export (SURVEY 8 f2): label list / classic indices against the pinned oracle, and the on-disk
layout of traindataexporter.cpp (dataset names, dtypes, chunking, result / plys bookkeeping)."""
import ctypes
import json
import os

import numpy as np
import pytest

from crazyara_b200.export import BLACK_WIN, DRAWN, WHITE_WIN, TrainDataExporter, read_dataset
from crazyara_b200.labels import classic_index, mirror_uci, uci_labels
from oracle.chess import Position, lib


@pytest.mark.parametrize("mode,n", [("crazyhouse", 2272), ("chess", 1968), ("lichess", 2316)])
def test_label_list_equals_oracle(mode, n):
    L = lib()
    L.opolicy_label.restype = ctypes.c_char_p
    m = {"crazyhouse": 0, "chess": 1, "lichess": 2}[mode]
    labels = uci_labels(mode)
    assert len(labels) == n == L.opolicy_nb_labels(m)
    assert labels == [L.opolicy_label(m, i).decode() for i in range(n)]


def test_classic_index_of_legal_moves_equals_oracle():
    L = lib()
    cases = [("crazyhouse", "crazyhouse", None, ["e2e4", "d7d5", "e4d5", "d8d5", "b1c3"]),
             ("chess", "chess", "r3k2r/pPpp1ppp/8/8/8/8/PPP2PpP/R3K2R w KQkq - 0 1", ["b7a8q"]),
             ("kingofthehill", "lichess", None, ["e2e4", "e7e5"])]
    checked = 0
    for variant, mode, fen, moves in cases:
        pos = Position(fen, variant, False)
        m = {"crazyhouse": 0, "chess": 1, "lichess": 2}[mode]
        for step in [None] + moves:
            if step is not None:
                pos.push_uci(step)
            black = pos.side_to_move() == 1
            for mv, uci in zip(pos.legal_moves(), pos.legal_uci()):
                want = L.opolicy_move_index(pos._buf, mv, m, 0)
                assert classic_index(mode, uci, black) == want, (uci, black)
                checked += 1
    assert checked > 150 and mirror_uci("e7e8q") == "e2e1q" and mirror_uci("N@f3") == "N@f6"


def test_exporter_layout_and_bookkeeping(tmp_path):
    path = str(tmp_path / "data.zarr")
    ex = TrainDataExporter(path, "crazyhouse", channels=34, number_chunks=3, chunk_size=4)
    rng = np.random.default_rng(0)
    games = []
    for g, (n, result) in enumerate([(3, WHITE_WIN), (5, BLACK_WIN), (2, DRAWN)]):
        game = ex.new_game()
        for i in range(n):
            planes = rng.integers(0, 3, (34, 8, 8)).astype(np.float32)
            stm = i & 1
            ex.save_sample(game, planes, ["e2e4", "N@f3"] if stm == 0 else ["e7e5", "N@f6"], [0.75, 0.25], 0.1 * i, stm)
        games.append((n, result, [x.copy() for x in game["x"]]))
        assert ex.export_game_samples(game, result) == n
    assert json.load(open(os.path.join(path, ".zgroup"))) == {"zarr_format": 2}
    meta = json.load(open(os.path.join(path, "x", ".zarray")))
    assert meta["shape"] == [12, 34, 8, 8] and meta["chunks"] == [4, 34, 8, 8] and meta["dtype"] == "<i2" and meta["compressor"] is None
    assert json.load(open(os.path.join(path, "y_policy", ".zarray")))["shape"] == [12, 2272]
    x = read_dataset(path, "x")
    assert x.dtype == np.int16 and np.array_equal(x[3], games[1][2][0]) and np.array_equal(x[9], games[2][2][1])
    v = read_dataset(path, "y_value")
    assert v[:3].tolist() == [1, -1, 1]            # white won: +1 for white to move
    assert v[3:8].tolist() == [-1, 1, -1, 1, -1]   # black won
    assert v[8:10].tolist() == [0, 0]
    assert read_dataset(path, "plys_to_end")[:10].tolist() == [3, 2, 1, 5, 4, 3, 2, 1, 2, 1]
    assert read_dataset(path, "start_indices")[:4].tolist() == [0, 3, 8, 10]
    pol = read_dataset(path, "y_policy")
    e2e4, nf3 = uci_labels("crazyhouse").index("e2e4"), uci_labels("crazyhouse").index("N@f3")
    assert pol[0, e2e4] == np.float32(0.75) and pol[0, nf3] == np.float32(0.25) and pol[0].sum() == 1.0
    assert pol[1, e2e4] == np.float32(0.75) and pol[1, nf3] == np.float32(0.25)  # black's e7e5 / N@f6 mirrored
    assert np.allclose(read_dataset(path, "y_best_move_q")[3:8], [0.0, 0.1, 0.2, 0.3, 0.4])
    # the file holds 12 samples: a game that does not fit is truncated, then the file is full
    game = ex.new_game()
    for i in range(5):
        ex.save_sample(game, np.zeros((34, 8, 8), np.float32), ["e2e4"], [1.0], 0.0, 0)
    assert ex.export_game_samples(game, DRAWN) == 2 and ex.is_file_full()


@pytest.mark.gpu
def test_arena_exports_samples(tmp_path):
    from crazyara_b200.engine import BoardState
    from crazyara_b200.selfplay import Arena, rl_settings
    from oracle import chess as ochess
    st = rl_settings("crazyhouse", batch_size=8, nodes=60, simulations=240)
    ex = TrainDataExporter(str(tmp_path / "sp.zarr"), "crazyhouse", channels=34, number_chunks=4, chunk_size=16)
    arena = Arena(None, st, variant=1, n_games=4, temperature_moves=4, max_plies=10, seed=2, exporter=ex)
    arena.run(min_games=4, max_steps=12)
    arena.close()
    path = str(tmp_path / "sp.zarr")
    assert ex.game_idx >= 4 and ex.start_idx >= 40
    starts = read_dataset(path, "start_indices")[:ex.game_idx + 1]
    assert starts[0] == 0 and np.all(np.diff(starts) > 0) and starts[-1] == ex.start_idx
    x = read_dataset(path, "x")
    want = ochess.planes(Position(None, "crazyhouse", False), "crazyhouse", 1, False).astype(np.int16)
    for s in starts[:-1]:
        assert np.array_equal(x[s], want)  # every game starts from the start position (un-normalised planes)
    pol = read_dataset(path, "y_policy")[:ex.start_idx]
    assert np.allclose(pol.sum(1), 1.0, atol=1e-5)
    plys = read_dataset(path, "plys_to_end")
    assert plys[starts[1] - 1] == 1 and plys[0] == starts[1]


def test_chess960_start_positions():
    """chess960fen (chess960position.h:36-80): all 960 arrangements are reachable, each is a legal chess960 set-up that
    the state code accepts with both castling rights per side."""
    import numpy as np
    from crazyara_b200.engine import BoardState
    from crazyara_b200.selfplay import chess960_fen
    rng = np.random.default_rng(7)
    seen = set()
    for _ in range(20000):
        fen = chess960_fen(rng)
        rank = fen.split("/")[7].split(" ")[0]
        seen.add(rank)
    assert len(seen) == 960 and "RNBQKBNR" in seen
    for rank in sorted(seen)[::37]:
        b = [i for i, c in enumerate(rank) if c == "B"]
        r = [i for i, c in enumerate(rank) if c == "R"]
        assert sorted(rank) == sorted("RNBQKBNR") and (b[0] + b[1]) % 2 == 1 and r[0] < rank.index("K") < r[1]
        st = BoardState().set(f"{rank.lower()}/pppppppp/8/8/8/8/PPPPPPPP/{rank} w KQkq - 0 1", True, 0)
        back = st.fen().split(" ")
        assert back[0].split("/")[7] == rank and len(back[2]) == 4      # four castling rights (Shredder letters)
        assert len(st.legal_actions()) >= 16                             # 16 pawn moves + knight moves


def test_selfplay_launcher_plan():
    """One worker per GPU: the concurrent games are split evenly, every worker writes the reference's file names
    (selfplay.cpp:116-127) and draws from its own seed range."""
    from crazyara_b200.selfplay import plan_workers
    plan = plan_workers(64, [0, 1, 2, 3, 4, 5, 6, 7], "/data/rl")
    assert [j["n_games"] for j in plan] == [8] * 8 and [j["device"] for j in plan] == list(range(8))
    assert plan[3]["zarr"] == "/data/rl/data_gpu_3.zarr" and plan[3]["pgn"] == "/data/rl/games_gpu_3.pgn"
    assert [j["seed_offset"] for j in plan] == list(range(0, 64, 8))
    uneven = plan_workers(10, [4, 5, 6], "o")
    assert [j["n_games"] for j in uneven] == [4, 3, 3] and sum(j["n_games"] for j in uneven) == 10
    assert [j["device"] for j in plan_workers(2, [0, 1, 2], "o")] == [0, 1]          # no idle worker is started


def test_chess960_generator_covers_the_reference_set():
    """The reference's chess960fen() (compiled from chess960position.h into oracle/_ref) reaches exactly 960 set-ups over
    30 000 seeds (tests/golden/ref_misc.json); ours must reach the same set, in the same FEN shape."""
    import json
    import os
    import numpy as np
    from crazyara_b200.selfplay import chess960_fen
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "ref_misc.json")))
    ref = g["chess960_back_ranks"]
    assert len(ref) == 960
    rng = np.random.default_rng(99)
    fens = {chess960_fen(rng) for _ in range(30000)}
    assert sorted(f.split("/")[7].split(" ")[0] for f in fens) == ref
    shape = sorted({f.split("/", 1)[1].split("/", 6)[0] + "|" + f.split(" ", 1)[1] for f in fens})
    assert shape == g["chess960_fen_shape"] == ["pppppppp|w KQkq - 0 1"]
    assert all(f.split("/")[0] == f.split("/")[7].split(" ")[0].lower() for f in fens)


def test_rl_settings_follow_the_reference_rl_config():
    """rl_settings / Arena defaults against the values of the reference's own UCIConfig dataclass
    (DeepCrazyhouse/configs/rl_config.py), recorded in tests/golden/rl_config.json."""
    import json
    import os
    cfg = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "rl_config.json")))
    import inspect
    from crazyara_b200.selfplay import Arena, rl_settings
    s = rl_settings("crazyhouse")
    assert s.batch_size == cfg["Batch_Size"] and s.nodes == cfg["Nodes"] and s.simulations == cfg["Simulations"]
    assert round(s.dirichlet_alpha * 100) == cfg["Centi_Dirichlet_Alpha"]
    assert round(s.dirichlet_epsilon * 100) == cfg["Centi_Dirichlet_Epsilon"]
    assert round(s.node_policy_temperature * 100) == cfg["Centi_Node_Temperature"]
    assert round(s.q_value_weight * 100) == cfg["Centi_Q_Value_Weight"] and bool(s.mcts_solver) == cfg["MCTS_Solver"]
    defaults = {k: v.default for k, v in inspect.signature(Arena.__init__).parameters.items()}
    assert round(defaults["temperature"] * 100) == cfg["Centi_Temperature"]
    assert defaults["temperature_moves"] == cfg["Temperature_Moves"] and defaults["reuse_tree"] == bool(cfg["Reuse_Tree"])
    from crazyara_b200.export import TrainDataExporter
    assert inspect.signature(TrainDataExporter.__init__).parameters["chunk_size"].default == cfg["Selfplay_Chunk_Size"]

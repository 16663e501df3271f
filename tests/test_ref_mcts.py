"""Pins the search oracle (oracle/mcts.c) to the REFERENCE'S OWN CODE.

`make -C oracle ref` compiles the reference's search sources unchanged -- node.cpp, nodedata.cpp, searchthread.cpp,
agents/mctsagent.cpp, agents/agent.cpp, evalinfo.cpp, manager/*.cpp, util/blazeutil.h, the settings structs -- into
oracle/_ref/libref_mcts.so, over three stand-ins for what the tree lacks: oracle/ref/blaze/Math.h (blaze-lib),
oracle/ref/pommermanstate.h (the environment: a `State` over oracle/chess.c, planes.c, policy.c) and a NeuralNetAPI
subclass that calls back into Python.  tests/golden/gen_ref_mcts_golden.py runs MCTSAgent::evaluate_board_state there for
every case below and records the results in tests/golden/ref_mcts.json; each case runs oracle/mcts.c here on the same
position, settings and network and demands IDENTICAL bits: visit counts, Q values, priors, MCTS posterior, root value,
best-move Q, node counters -- at node temperature 1 and 1.7 (std::pow -> glibc powf), with Dirichlet noise (the real
std::gamma_distribution over std::default_random_engine), with the MCTS solver on mate positions, in every virtual-loss
style.

What stays a stand-in, and is therefore NOT pinned by this: blaze's evaluation of get_current_u_values
((v*s)*w restructured to (v*w)*s, see blaze/Math.h), blaze::sum's reduction order, and the order of Stockfish's move
generator (the environment returns moves in ascending policy-index order).

The network is oracle.search.hash_net (tie-free priors): with oracle/fake.c's 2048-level priors tied moves are common
and std::sort's unspecified order among them (node.cpp:464-470) would be compared, not the search."""
import functools
import json
import os

import numpy as np
import pytest

from oracle import search as osr
from oracle.chess import Position
from tests.test_search_hostemu import CASES, case_settings

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_mcts.json")


def _bits(a):
    return np.asarray(a, np.float32).view(np.uint32)


@functools.lru_cache(maxsize=None)
def _golden():
    with open(GOLDEN) as f:
        return json.load(f)


def _ids(cases):
    return [f"{c[0]}-b{c[6]}-s{c[7]}-{i}" for i, c in enumerate(cases)]


def _fixed(case, **extra):
    """(position, fen, variant id, chess960, premoves, settings) of a CASES row."""
    variant, vid, mode, fen, is960, premoves, batch, sims, row_extra = case
    st = case_settings(mode, batch, sims, dict(row_extra, **extra))
    pos = Position(fen, variant, is960)
    pos.push_uci(*premoves)
    return pos, fen, vid, is960, premoves, st


def _random(seed):
    """The randomised positions / settings of tests/test_search_fuzz_hostemu.py (all four variants, random temperature,
    Dirichlet, virtual styles, solver on/off, node limits)."""
    from tests.test_search_fuzz_hostemu import VARIANTS, _random_case
    pos, _, st, (vid, played) = _random_case(seed)
    root = Position(None, VARIANTS[seed % len(VARIANTS)][0], False)
    root.push_uci(*played)
    assert root.fen() == pos.fen()
    return pos, None, vid, False, played, st


# Threads = 2: the reference counts the virtual visits in flight on an edge in a uint8 (nodedata.h:93, asserted in
# node.h:506), so Batch_Size x Threads must stay below 256 -- the B = 128 cases cannot run with two threads there
CASES_2T = [c for c in CASES if 2 * c[6] < 256]

EPS = dict(epsilon_greedy_counter=20, epsilon_checks_counter=100)  # the UCI defaults Centi_Epsilon_Greedy 5, _Checks 1


def searches():
    """(golden key, search set-up, threads) of every comparison below: what gen_ref_mcts_golden.py records."""
    for cid, case in zip(_ids(CASES), CASES):
        yield f"threads1/{cid}", _fixed(case), 1
    for seed in range(24):
        yield f"random/{seed}", _random(seed), 1
    for cid, case in zip(_ids(CASES_2T), CASES_2T):
        yield f"threads2/{cid}", _fixed(case, threads=2), 2
    for threads in (1, 2):
        for cid, case in zip(_ids(CASES_2T), CASES_2T):
            yield f"epsilon{threads}/{cid}", _fixed(case, threads=threads, **EPS), threads


def assert_oracle_equals_reference(key, setup, threads):
    pos, _fen, _vid, _is960, _premoves, st = setup
    S = osr.Search(st)
    ro = S.run(pos, osr.hash_net(S.n_labels), with_keys=True, threads=threads)
    rr = _golden()[key]
    assert ro["visit_sum"] > 0
    assert ro["moves"] == rr["moves"]                      # same prior order (no ties with this network)
    assert np.array_equal(ro["visits"], np.array(rr["visits"], np.uint32))
    k = rr["no_visit_idx"]                                 # the reference holds Q only for the children opened so far
    assert k == int(np.count_nonzero(ro["visits"])) or k >= int(np.count_nonzero(ro["visits"]))
    assert np.array_equal(_bits(ro["q"][:k]), np.array(rr["q_bits"][:k], np.uint32))
    assert np.array_equal(_bits(ro["prior"]), np.array(rr["prior_bits"], np.uint32))
    assert np.array_equal(ro["policy"][:len(rr["policy"])], np.array(rr["policy"], np.float64))
    for name in ("visit_sum", "free_visits", "nodes", "root_value", "best_move_q"):
        assert ro[name] == rr[name], name
    assert ro["moves"][ro["best_idx"]] == rr["moves"][rr["best_idx"]]


@pytest.mark.parametrize("cid,case", list(zip(_ids(CASES), CASES)), ids=_ids(CASES))
def test_oracle_search_equals_the_compiled_reference_search(cid, case):
    assert_oracle_equals_reference(f"threads1/{cid}", _fixed(case), 1)


@pytest.mark.parametrize("seed", range(24))
def test_oracle_search_equals_the_compiled_reference_search_on_random_cases(seed):
    assert_oracle_equals_reference(f"random/{seed}", _random(seed), 1)


@pytest.mark.parametrize("cid,case", list(zip(_ids(CASES_2T), CASES_2T)), ids=_ids(CASES_2T))
def test_oracle_two_thread_schedule_equals_the_compiled_reference_search(cid, case):
    """Threads = 2 (the reference's default): two SearchThread objects of the compiled reference driven in the fixed
    schedule of oracle/mcts.h -- sel(0) sel(1) | bk(0) sel(0) bk(1) sel(1) | ... , one of the interleavings its two OS
    threads can produce -- against the oracle's two logical threads in the same schedule: identical bits."""
    assert_oracle_equals_reference(f"threads2/{cid}", _fixed(case, threads=2), 2)


def test_glibc_rand_restatement_equals_libc():
    """oracle/mcts.c restates glibc's rand() (the exploration branches draw `rand() % counter`); the device code restates it
    again (search_dev.cuh): both pinned to the live libc here / in tests/test_glibc_flt32.py."""
    import ctypes
    L = osr._lib()
    libc = ctypes.CDLL("libc.so.6")
    for seed in (1, 42, 0, 123456789, 2**32 - 1):
        out = np.zeros(2000, np.int32)
        L.oglibc_rand_sequence(seed, len(out), out.ctypes.data)
        libc.srand(seed)
        assert [libc.rand() for _ in range(len(out))] == out.tolist()


@pytest.mark.parametrize("threads", [1, 2])
@pytest.mark.parametrize("cid,case", list(zip(_ids(CASES_2T), CASES_2T)), ids=_ids(CASES_2T))
def test_epsilon_exploration_equals_the_compiled_reference_search(cid, case, threads):
    """Centi_Epsilon_Greedy 5 / Centi_Epsilon_Checks 1 (the reference's UCI defaults, optionsuci.cpp:89-90): random
    playouts and unexplored checks below a randomly deep node of the main line (searchthread.cpp:124-185, :451-473),
    driven by the C library's rand() seeded with the settings' seed."""
    assert_oracle_equals_reference(f"epsilon{threads}/{cid}", _fixed(case, threads=threads, **EPS), threads)

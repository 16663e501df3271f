"""Generates tests/golden/ref_mcts.json: the reference's own search (oracle/_ref/libref_mcts.so, `make -C oracle ref`,
which needs the reference's engine sources) on every case of tests/test_ref_mcts.py.  Q values and priors are stored as
float32 bit patterns, so the test compares bits.  Run where oracle/_ref has been built:
    python tests/golden/gen_ref_mcts_golden.py"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)


def main():
    from oracle import refmcts
    from oracle import search as osr
    from tests.test_ref_mcts import searches
    out = {}
    for key, (pos, fen, vid, is960, premoves, st), _threads in searches():
        S = osr.Search(st)
        rr = refmcts.run(pos, fen, vid, is960, premoves, st, net_fn=osr.hash_net(S.n_labels), channels=S.channels,
                         n_labels=S.n_labels)
        S.close()
        k = rr["no_visit_idx"]
        out[key] = dict(moves=rr["moves"], visits=rr["visits"].tolist(), no_visit_idx=k,
                        q_bits=rr["q"][:k].view(np.uint32).tolist(), prior_bits=rr["prior"].view(np.uint32).tolist(),
                        policy=rr["policy"].tolist(), visit_sum=rr["visit_sum"], free_visits=rr["free_visits"],
                        nodes=rr["nodes"], root_value=rr["root_value"], best_move_q=rr["best_move_q"],
                        best_idx=rr["best_idx"])
    with open(os.path.join(HERE, "ref_mcts.json"), "w") as f:
        json.dump(out, f, separators=(",", ":"))
    print(len(out), "searches")


if __name__ == "__main__":
    main()

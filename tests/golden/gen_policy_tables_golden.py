"""Generates tests/golden/policy_tables_reference.json: the reference's frozen label lists (engine/tests/legacyconstants.h)
and FLAT_PLANE_IDX tables (engine/src/environments/chess_related/policymaprepresentation.h), read from a CrazyAra
checkout:
    python tests/golden/gen_policy_tables_golden.py <CrazyAra checkout>"""
import json
import os
import re
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ORDER = (("crazyhouse", 0), ("lichess", 1), ("chess", 2))  # order of the tables in both headers


def main(checkout):
    engine = os.path.join(checkout, "engine")
    src = open(os.path.join(engine, "src/environments/chess_related/policymaprepresentation.h")).read()
    parts = re.split(r"const unsigned long FLAT_PLANE_IDX\[\] = \{", src)[1:]
    tabs = [[int(x) for x in re.findall(r"\d+", p.split("};")[0])] for p in parts]
    leg = open(os.path.join(engine, "tests/legacyconstants.h")).read()
    lists = [re.findall(r'"([^"]+)"', b.split("};")[0]) for b in re.split(r"const std::string LABELS\[\] = \{", leg)[1:]]
    out = {name: {"labels": ",".join(lists[i]), "flat_plane_idx": tabs[i]} for name, i in ORDER}
    with open(os.path.join(HERE, "policy_tables_reference.json"), "w") as f:
        json.dump(out, f, separators=(",", ":"))
    print({name: len(lists[i]) for name, i in ORDER})


if __name__ == "__main__":
    main(sys.argv[1])

"""Generates tests/golden/rl_config.json: the field values of the reference's UCIConfig dataclass
(DeepCrazyhouse/configs/rl_config.py), read from a CrazyAra checkout:
    python tests/golden/gen_rl_config_golden.py <CrazyAra checkout>"""
import importlib.util
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))


def main(checkout):
    spec = importlib.util.spec_from_file_location("ref_rl_config", os.path.join(checkout, "DeepCrazyhouse", "configs",
                                                                               "rl_config.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    with open(os.path.join(HERE, "rl_config.json"), "w") as f:
        json.dump(dict(vars(mod.UCIConfig())), f, indent=1, sort_keys=True)


if __name__ == "__main__":
    main(sys.argv[1])

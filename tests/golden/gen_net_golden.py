"""Generates tests/golden/net_<arch>.json by running the REAL reference network definition
(/root/reference/DeepCrazyhouse/src/domain/neural_net/architectures/pytorch/rise_mobile_v3.py) on the seeded
state_dict of oracle/net.py.  Run in the build container only (the GPU box has no /root/reference):
    python tests/golden/gen_net_golden.py
"""
import json
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import net as onet  # noqa: E402


def load_reference_models():
    timm, tm, tl = types.ModuleType("timm"), types.ModuleType("timm.models"), types.ModuleType("timm.models.layers")

    class DropPath(torch.nn.Module):  # identity: only used with path_dropout=0
        def __init__(self, p=0.0):
            super().__init__()

        def forward(self, x):
            return x

    tl.DropPath = DropPath
    tl.trunc_normal_ = lambda *a, **k: None
    sys.modules.update({"timm": timm, "timm.models": tm, "timm.models.layers": tl})
    sys.path.insert(0, "/root/reference")
    from DeepCrazyhouse.src.domain.neural_net.architectures.pytorch.rise_mobile_v3 import (get_rise_v2_model,
                                                                                             get_rise_v33_model)
    return get_rise_v2_model, get_rise_v33_model


def reference_forward(arch, sd_np, x):
    get_v2, get_v33 = load_reference_models()

    class Args:
        pass

    a = Args()
    a.input_shape = (arch["in_channels"], 8, 8)
    a.channels_policy_head = arch["policy_channels"]
    a.select_policy_from_plane = True
    a.n_labels = 2272
    a.use_wdl = a.use_plys_to_end = arch["wdl"]
    a.use_mlp_wdl_ply = False
    model = (get_v2 if arch["name"] == "risev2" else get_v33)(a)
    sd = model.state_dict()
    missing = [k for k in sd if k not in sd_np and not k.endswith("num_batches_tracked")
               and not (arch["wdl"] and k.startswith("value_head.body_final"))]
    assert not missing, missing
    for k, v in sd_np.items():
        assert tuple(sd[k].shape) == tuple(v.shape), (k, sd[k].shape, v.shape)
        sd[k] = torch.from_numpy(v)
    model.load_state_dict(sd)
    model.eval()
    with torch.no_grad():
        out = model(torch.from_numpy(x))
    value, logits = out[0].numpy()[:, 0], out[1].numpy()
    aux = out[2].numpy() if arch["wdl"] else None
    return value, logits, aux


def golden_input(arch, n=4, seed=123):
    rng = np.random.default_rng(seed)
    x = (rng.random((n, arch["in_channels"], 8, 8)) < 0.15).astype(np.float32)
    x[:, -3:] = rng.random((n, 3, 1, 1)).astype(np.float32)  # a few scalar planes
    return x


def _f32(a):
    """float32 values as the shortest decimals that read back to the same float32."""
    return [float(f"{x:.9g}") for x in np.asarray(a, np.float32).ravel()]


def record_live_cases():
    """tests/golden/net_reference_live.json: the reference module on state_dict seed 7 and three input positions (seed 9)
    for the architectures test_oracle_net_matches_imported_reference checks; the logits at every 11th column plus the
    sums over all columns."""
    rec = {}
    for name, arch in (("risev2_34", onet.arch_risev2(34, 81)), ("risev33_52", onet.arch_risev33(52, 76, True))):
        sd = onet.make_state_dict(arch, 7)
        value, logits, aux = reference_forward(arch, sd, golden_input(arch, n=3, seed=9))
        idx = np.arange(0, logits.shape[1], 11)
        rec[name] = dict(seed=7, input_seed=9, n=3, value=_f32(value), aux=None if aux is None else _f32(aux),
                         logit_idx=idx.tolist(), logits=_f32(logits[:, idx]), logits_sum=logits.astype(np.float64).sum(1).tolist(),
                         logits_abs_sum=np.abs(logits.astype(np.float64)).sum(1).tolist())
    path = os.path.join(ROOT, "tests", "golden", "net_reference_live.json")
    with open(path, "w") as f:
        json.dump(rec, f, separators=(",", ":"))
    print("wrote", path)


def main():
    for arch in (onet.arch_risev2(34, 81), onet.arch_risev33(52, 76, True), onet.arch_risev2(63, 84)):
        sd = onet.make_state_dict(arch, seed=0)
        x = golden_input(arch)
        value, logits, aux = reference_forward(arch, sd, x)
        prob = torch.softmax(torch.from_numpy(logits), dim=1).numpy()
        idx = np.arange(0, logits.shape[1], 97)
        rec = dict(arch=arch["name"], in_channels=arch["in_channels"], policy_channels=arch["policy_channels"],
                   seed=0, input_seed=123, value=value.tolist(), aux=None if aux is None else aux.tolist(),
                   logit_idx=idx.tolist(), logits=logits[:, idx].tolist(), prob=prob[:, idx].tolist(),
                   logits_sum=logits.sum(1).tolist(), logits_abs_sum=np.abs(logits).sum(1).tolist(),
                   argmax=logits.argmax(1).tolist())
        path = os.path.join(ROOT, "tests", "golden", f"net_{arch['name']}_{arch['in_channels']}.json")
        with open(path, "w") as f:
            json.dump(rec, f)
        print("wrote", path, "value", value)
    record_live_cases()


if __name__ == "__main__":
    main()

"""TEST INFRASTRUCTURE — golden fixture for the ResNet-101 zero-shot model from the REAL reference.

Runs only where the reference tree is available (build container): constructs the unmodified reference
`LSegRNNetZS(label_list, backbone="clip_resnet101", ...)` (modules/models/lseg_net_zs.py:240-378: torchvision resnet101
split into pretrained.layer1..4 by _make_resnet_backbone, the scratch decoder, the per-image ['others', name] head),
loads the seeded state dict (oracle/synth.py, backbone="clip_resnet101"), runs it on seeded inputs, checks that the
oracle restatement (oracle/lseg_oracle.py::lseg_forward_rn_zs — torchvision's Bottleneck restated) reproduces it (the
ResNet stages and path_1 to 1e-5, logits within the fp16 text-tower floor), and writes tests/golden/ref_rn101.npz and
tests/golden/state_dict_keys_rn101.json.

Usage:  LSEG_REFERENCE_ROOT=<lang-seg checkout> python oracle/make_golden_rn.py
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import lseg_oracle as O  # noqa: E402
from oracle import ref_standins as R  # noqa: E402
from oracle import synth  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
BACKBONE = "clip_resnet101"


def _stats(t):
    t = t.detach().float()
    return np.array([t.mean().item(), t.std().item(), t.abs().max().item()], dtype=np.float64)


def _rel(a, b):
    return ((a - b).abs().max() / (a.abs().max() + 1e-12)).item()


def main():
    torch.set_num_threads(os.cpu_count() or 1)
    sd = synth.make_state_dict(0, backbone=BACKBONE)
    names = [line.strip() for line in open(os.path.join(GOLD, "fewshot_pascal.txt")) if line.strip()]
    R.install()
    cwd = os.getcwd()
    os.chdir(R.REFERENCE_ROOT)
    try:
        from modules.models.lseg_net_zs import LSegRNNetZS
        net = LSegRNNetZS(label_list=names, backbone=BACKBONE, features=256, arch_option=0, block_depth=0,
                          activation="lrelu", use_pretrained=False)
    finally:
        os.chdir(cwd)
    missing, unexpected = net.load_state_dict(sd, strict=False)
    missing = [k for k in missing if "num_batches_tracked" not in k]
    assert not missing and not unexpected, (missing[:5], unexpected[:5])
    net.eval()
    with open(os.path.join(GOLD, "state_dict_keys_rn101.json"), "w") as f:
        json.dump({k: list(v.shape) for k, v in net.state_dict().items()}, f, indent=0, sort_keys=True)
    cap = {}
    for k in range(4):
        getattr(net.scratch, f"layer{k + 1}_rn").register_forward_hook(
            lambda m, a, o, k=k: cap.__setitem__(f"layer{k}", a[0].detach()))
    net.scratch.refinenet1.register_forward_hook(lambda m, a, o: cap.__setitem__("path1", o.detach()))
    texts = [synth.tokenize(["others", n]) for n in names]
    out = {}
    for tag, (B, H, W, seed) in {"small": (3, 96, 128, 77), "s480": (2, 480, 480, 1480)}.items():
        x = synth.make_image(B, H, W, seed=seed)
        class_info = torch.tensor([3, 0, 17][:B])
        with torch.no_grad():
            ref = net(x, class_info)
        got, st = O.lseg_forward_rn_zs(x, class_info, texts, sd, return_stages=True)
        for k in range(4):
            e = _rel(cap[f"layer{k}"], st["layers"][k])
            assert e < 1e-5, (tag, k, e)
        e1 = _rel(cap["path1"], st["path_1"])
        e2 = _rel(ref, got)
        print(f"{tag}: oracle vs reference path1 {e1:.2e}, logits {e2:.2e} (two fp16 text-tower executions), "
              f"argmax {(ref.argmax(1) == got.argmax(1)).float().mean().item():.4f}")
        assert e1 < 1e-5 and e2 < 5e-3
        out[f"{tag}_class_info"] = class_info.numpy()
        out[f"{tag}_floor"] = np.array(e2)
        out[f"{tag}_layers_stats"] = np.stack([_stats(cap[f"layer{k}"]) for k in range(4)])
        out[f"{tag}_path1_stats"] = _stats(cap["path1"])
        if tag == "small":
            out["small_logits"] = ref.numpy()
        else:
            out["s480_logits_lattice"] = ref[:, :, ::4, ::4].numpy()
            out["s480_argmax"] = ref.argmax(1).to(torch.uint8).numpy()
            top2 = ref.topk(2, dim=1).values
            out["s480_margin_f16"] = (top2[:, 0] - top2[:, 1]).half().numpy()
    np.savez_compressed(os.path.join(GOLD, "ref_rn101.npz"), **out)
    print("written tests/golden/ref_rn101.npz")


if __name__ == "__main__":
    main()

"""TEST INFRASTRUCTURE — golden fixtures for the non-default backbones from the REAL reference.

Runs only where the reference tree is available (build container). For
  * clip_vitb32_384 (lseg_net.py:119-123 hooks 2/5/8/11; lseg_vit.py:259-405: timm vit_base_patch32_384, reassemble to
    96/192/384/768 channels with ConvTranspose x8 / x4 / x2 / none; CLIP ViT-B/32 text tower)        -> tag "b32"
  * clipRN50x16_vitl16_384 (lseg_vit.py:240-257: the ViT-L/16 trunk with CLIP RN50x16's text tower — width 768, 12 heads,
    embedding 768 = out_c, lseg_net.py:142-146)                                                        -> tag "rn50x16"
it constructs the unmodified reference LSegNet, loads the seeded state dict (oracle/synth.py, backbone=...), runs it on
seeded inputs, checks that the oracle restatement reproduces it (image trunk to 1e-5, logits within the fp16 text-tower
floor), and writes tests/golden/ref_<tag>.npz and tests/golden/state_dict_keys_<tag>.json (key -> shape contract).

Usage:  LSEG_REFERENCE_ROOT=<lang-seg checkout> python oracle/make_golden_backbones.py [b32] [rn50x16]
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

TAGS = {"b32": "clip_vitb32_384", "rn50x16": "clipRN50x16_vitl16_384"}


def _stats(t):
    t = t.detach().float()
    return np.array([t.mean().item(), t.std().item(), t.abs().max().item()], dtype=np.float64)


def _rel(a, b):
    return ((a - b).abs().max() / (a.abs().max() + 1e-12)).item()


def make(TAG, BACKBONE):
    sd = synth.make_state_dict(0, backbone=BACKBONE)
    ade = synth.ade20k_labels()
    net = R.build_reference_net(sd, ade, backbone=BACKBONE)
    with open(os.path.join(ROOT, "tests", "golden", f"state_dict_keys_{TAG}.json"), "w") as f:
        json.dump({k: list(v.shape) for k, v in net.state_dict().items()}, f, indent=0, sort_keys=True)
    cap = {}
    for i, blk in enumerate(O.BACKBONES[BACKBONE]["hooks"]):
        net.pretrained.model.blocks[blk].register_forward_hook(lambda m, a, o, i=i: cap.__setitem__(f"tap{i}", o.detach()))
    for k in range(4):
        getattr(net.scratch, f"layer{k + 1}_rn").register_forward_hook(
            lambda m, a, o, k=k: cap.__setitem__(f"layer{k}", a[0].detach()))
    net.scratch.refinenet1.register_forward_hook(lambda m, a, o: cap.__setitem__("path1", o.detach()))
    out = {}
    for tag, (B, H, W, labels, seed) in {"small": (2, 64, 96, ade[:5], 2064), "k150": (1, 480, 480, ade, 1480)}.items():
        x = synth.make_image(B, H, W, seed=seed)
        with torch.no_grad():
            ref = net(x, labels)
        got, st = O.lseg_forward(x, synth.tokenize(labels), sd, return_stages=True, backbone=BACKBONE)
        for i in range(4):
            e = _rel(cap[f"tap{i}"], st["taps"][i])
            assert e < 1e-5, (tag, "tap", i, e)
            e = _rel(cap[f"layer{i}"], st["layers"][i])
            assert e < 1e-5, (tag, "layer", i, e)
        e1 = _rel(cap["path1"], st["path_1"])
        e2 = _rel(ref, got)
        agree = (ref.argmax(1) == got.argmax(1)).float().mean().item()
        print(f"{TAG} {tag}: oracle vs reference path1 {e1:.2e}, logits {e2:.2e} (two fp16 text-tower executions), argmax {agree:.4f}")
        assert e1 < 1e-5 and e2 < 5e-3  # floor of two executions of the chaotic fp16 text tower (tests/test_oracle.py)
        top2 = ref.topk(2, dim=1).values
        if tag == "small":
            out["small_logits"] = ref.numpy()
            out["small_labels"] = np.array(labels)
        else:
            out["k150_logits_lattice"] = ref[:, :, ::8, ::8].numpy()
            out["k150_argmax"] = ref.argmax(1).to(torch.uint8).numpy()
            out["k150_margin_f16"] = (top2[:, 0] - top2[:, 1]).half().numpy()
        out[f"{tag}_floor"] = np.array(e2)  # the reference's two executions of its fp16 text tower, in the logits
        out[f"{tag}_taps_stats"] = np.stack([_stats(cap[f"tap{i}"]) for i in range(4)])
        out[f"{tag}_layers_stats"] = np.stack([_stats(cap[f"layer{i}"]) for i in range(4)])
        out[f"{tag}_path1_stats"] = _stats(cap["path1"])
        out[f"{tag}_tap3_row0"] = cap["tap3"][0, 0].numpy()
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", f"ref_{TAG}.npz"), **out)
    print(f"written tests/golden/ref_{TAG}.npz")


if __name__ == "__main__":
    torch.set_num_threads(os.cpu_count() or 1)
    for tag in (sys.argv[1:] or list(TAGS)):
        make(tag, TAGS[tag])

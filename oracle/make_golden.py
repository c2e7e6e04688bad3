"""TEST INFRASTRUCTURE — generate the golden fixtures under tests/golden/ from the REAL reference.

Runs only where a lang-seg checkout is named by LSEG_REFERENCE_ROOT: imports the reference's
modules/models/lseg_net.py unchanged through oracle/ref_standins.py, loads the seeded synthetic state
dict (oracle/synth.py), runs LSegNet.forward on seeded inputs, verifies that the oracle restatement
(oracle/lseg_oracle.py) reproduces it, and writes small fixtures:

  tests/golden/ref_small.npz    B=2, 64x96, K=5   : full logits (fp16-exact values stored as fp32), taps/path
                                                    checksums
  tests/golden/ref_480_k150.npz B=1, 480x480, K=150: logits at a stride-8 pixel lattice, full argmax mask
                                                    (uint8), text features, per-stage statistics
  tests/golden/ref_480_k2.npz   B=1, 480x480, ['cat','other'] (BASELINE.json configs[0])
  tests/golden/ref_zs.npz       zero-shot path (lseg_net_zs.py) B=3, 96x96, PASCAL label file
  tests/golden/state_dict_keys.json : key -> shape contract of the reference LSegNet

Usage:  LSEG_REFERENCE_ROOT=<lang-seg checkout> python oracle/make_golden.py
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


def _stats(t):
    t = t.detach().float()
    return np.array([t.mean().item(), t.std().item(), t.abs().max().item()], dtype=np.float64)


def _check(name, ref, got, tol):
    err = ((ref - got).abs().max() / (ref.abs().max() + 1e-12)).item()
    print(f"  oracle vs reference [{name}]: max rel err {err:.3e}")
    assert err <= tol, (name, err)
    return err


def main():
    torch.set_num_threads(os.cpu_count() or 1)
    sd = synth.make_state_dict(0)
    ade = synth.ade20k_labels()
    net = R.build_reference_net(sd, ade)

    # contract of state-dict keys (SURVEY.md Appendix C)
    keys = {k: list(v.shape) for k, v in net.state_dict().items()}
    with open(os.path.join(GOLD, "state_dict_keys.json"), "w") as f:
        json.dump(keys, f, indent=0, sort_keys=True)

    # hook the reference's own sub-modules to capture per-stage tensors
    cap = {}
    hooks = []
    for i, blk in enumerate((5, 11, 17, 23)):
        hooks.append(net.pretrained.model.blocks[blk].register_forward_hook(
            lambda m, a, o, i=i: cap.__setitem__(f"tap{i}", o.detach())))
    hooks.append(net.scratch.refinenet1.register_forward_hook(lambda m, a, o: cap.__setitem__("path1", o.detach())))

    def run_ref(x, labels):
        with torch.no_grad():
            return net(x, labels) if labels is not None else net(x)

    # ---- small ----
    labels5 = ade[:5]
    x = synth.make_image(2, 64, 96, seed=2064)
    ref = run_ref(x, labels5)
    got, st = O.lseg_forward(x, synth.tokenize(labels5), sd, return_stages=True)
    for i in range(4):
        _check(f"small tap{i}", cap[f"tap{i}"], st["taps"][i], 1e-5)
    _check("small path1", cap["path1"], st["path_1"], 1e-5)
    _check("small logits", ref, got, 3e-3)  # text tower: nn.MultiheadAttention vs restated MHA, both fp16
    np.savez_compressed(os.path.join(GOLD, "ref_small.npz"), logits=ref.numpy(),
                        taps_stats=np.stack([_stats(cap[f"tap{i}"]) for i in range(4)]),
                        path1_stats=_stats(cap["path1"]), tap3_row0=cap["tap3"][0, 0].numpy(),
                        labels=np.array(labels5))

    # ---- 480x480, K=150 (BASELINE.json configs[1] at B=1) and K=2 (configs[0]) ----
    for tag, labels in (("k150", ade), ("k2", ["cat", "other"])):
        x = synth.make_image(1, 480, 480, seed=1480)
        ref = run_ref(x, labels)
        got, st = O.lseg_forward(x, synth.tokenize(labels), sd, return_stages=True)
        _check(f"480 {tag} tap3", cap["tap3"], st["taps"][3], 1e-5)
        _check(f"480 {tag} path1", cap["path1"], st["path_1"], 1e-5)
        _check(f"480 {tag} logits", ref, got, 3e-3)
        agree = (ref.argmax(1) == got.argmax(1)).float().mean().item()
        print(f"  argmax agreement oracle vs reference: {agree:.6f}")
        with torch.no_grad():
            tf = net.clip_pretrained.encode_text(synth.tokenize(labels))
            tf = tf / tf.norm(dim=-1, keepdim=True)
        top2 = ref.topk(2, dim=1).values
        np.savez_compressed(os.path.join(GOLD, f"ref_480_{tag}.npz"),
                            logits_lattice=ref[:, :, ::8, ::8].numpy(),
                            argmax=ref.argmax(1).to(torch.uint8).numpy(),
                            margin_f16=(top2[:, 0] - top2[:, 1]).half().numpy(),
                            text_features=tf.numpy(),
                            taps_stats=np.stack([_stats(cap[f"tap{i}"]) for i in range(4)]),
                            path1_stats=_stats(cap["path1"]), tap3_row0=cap["tap3"][0, 0].numpy())

    # ---- zero-shot path ----
    for h in hooks:
        h.remove()
    cwd = os.getcwd()
    os.chdir(R.REFERENCE_ROOT)
    try:
        # lseg_net_zs.py imports its own *_zs block files, which pull extra backbones from timm/clip/torchvision
        import timm
        timm.create_model = lambda name, pretrained=False, **kw: R.VisionTransformer()
        from modules.models.lseg_net_zs import LSegNetZS
        names = [line.strip() for line in open(os.path.join(GOLD, "fewshot_pascal.txt")) if line.strip()]
        zs = LSegNetZS(label_list=names, backbone="clip_vitl16_384", features=256, arch_option=0, block_depth=0,
                       activation="lrelu")
    finally:
        os.chdir(cwd)
    zs.load_state_dict(sd, strict=False)
    zs.eval()
    x = synth.make_image(3, 96, 96, seed=77)
    class_info = torch.tensor([3, 0, 17])
    with torch.no_grad():
        ref = zs(x, class_info)
    texts = [synth.tokenize(["others", n]) for n in names]
    got = O.lseg_forward_zs(x, class_info, texts, sd)
    _check("zero-shot logits", ref, got, 3e-3)
    np.savez_compressed(os.path.join(GOLD, "ref_zs.npz"), logits=ref.numpy(), class_info=class_info.numpy())
    print("golden fixtures written to", GOLD)


if __name__ == "__main__":
    main()

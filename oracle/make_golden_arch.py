"""TEST INFRASTRUCTURE — golden fixture for the arch_option 1 / 2 head blocks from the REAL reference.

Runs only where the reference tree is available (build container): constructs the unmodified reference LSegNet with
arch_option 1 (bottleneck_block, block_depth 2, lrelu) and 2 (depthwise_block, block_depth 3, tanh), loads the seeded
state dict (oracle/synth.py, head_block=True), runs it on a seeded input, checks that the oracle restatement
(oracle/lseg_oracle.py::head_block) reproduces it, and writes tests/golden/ref_arch.npz.

Usage:  LSEG_REFERENCE_ROOT=<lang-seg checkout> python oracle/make_golden_arch.py
"""
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

CASES = {"opt1": dict(arch_option=1, block_depth=2, activation="lrelu"),
         "opt2": dict(arch_option=2, block_depth=3, activation="tanh")}


def main():
    torch.set_num_threads(os.cpu_count() or 1)
    sd = synth.make_state_dict(0, head_block=True)
    labels = synth.ade20k_labels()[:5]
    x = synth.make_image(2, 64, 96, seed=2064)
    out = {}
    for tag, kw in CASES.items():
        net = R.build_reference_net(sd, labels, **kw)
        with torch.no_grad():
            ref = net(x)
        got = O.lseg_forward(x, synth.tokenize(labels), sd, **kw)
        err = ((ref - got).abs().max() / ref.abs().max()).item()
        print(f"{tag}: oracle vs reference max rel err {err:.3e} (text tower: two fp16 executions)")
        assert err < 3e-2, err  # the blocks amplify the 2e-3 text-tower difference (3x3 taps up to 0.4, channel max)
        # the head block itself, on the reference's own pre-block logits: bit-level
        cap = {}
        h = net.scratch.head_block.register_forward_hook(lambda m, a, o: cap.setdefault("first_in", a[0].detach().clone()))
        with torch.no_grad():
            net(x)
        h.remove()
        blk = O.head_block(cap["first_in"], sd, **kw)
        with torch.no_grad():
            want = cap["first_in"]
            for _ in range(kw["block_depth"] - 1):
                want = net.scratch.head_block(want)
            want = net.scratch.head_block(want, False)
        assert torch.equal(blk, want), "oracle head_block differs from the reference module"
        out[f"{tag}_logits"] = ref.numpy()
        out[f"{tag}_pre_block"] = cap["first_in"].numpy()
        out[f"{tag}_post_block"] = want.numpy()
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "ref_arch.npz"), **out)
    print("written tests/golden/ref_arch.npz")


if __name__ == "__main__":
    main()

"""TEST INFRASTRUCTURE. Golden vectors for the multi-scale evaluator (SURVEY.md 8(f) row 1).

Runs the UNMODIFIED reference class `additional_utils/models.py::LSeg_MultiEvalModule.forward` on CPU — the only
intervention is `torch.Tensor.cuda = identity`, because the class hard-codes `.cuda()` on its accumulators — around a
small, exactly batch-invariant stand-in network (elementwise arithmetic only), and stores inputs, stand-in parameters
and outputs in tests/golden/ref_multiscale.npz. tests/test_evaluator_cpu.py replays them through
lseg_b200.evaluator.MultiScaleEvaluator.

    LSEG_REFERENCE_ROOT=<lang-seg checkout> python oracle/make_golden_eval.py
"""
import contextlib
import io
import os
import sys

import numpy as np
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class StandInNet(nn.Module):
    """net(x[B,3,c,c], label_set) -> [B,K,c,c]; elementwise ops only, so batch 1 and batch N agree bit for bit.
    Position dependent (pos) and not flip symmetric (the rolled term), so window placement and flips matter."""

    def __init__(self, K, crop, seed):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.Wc = torch.randn(K, 3, generator=g)
        self.V = torch.randn(K, generator=g)
        self.pos = torch.randn(1, K, crop, crop, generator=g) * 0.3

    def forward(self, x, label_set=""):
        outs = []
        for k in range(self.Wc.shape[0]):
            o = x[:, 0] * self.Wc[k, 0] + x[:, 1] * self.Wc[k, 1] + x[:, 2] * self.Wc[k, 2]
            o = o + 0.5 * torch.roll(x[:, 0], 1, dims=-1) * self.V[k]
            outs.append(o)
        return torch.stack(outs, 1) + self.pos


CASES = [  # (h, w, base_size, crop_size, scales, K, flip)
    (48, 40, 64, 32, [0.5, 0.75, 1.0, 1.25, 1.5, 1.75], 5, True),    # portrait, every branch of the size logic
    (40, 72, 64, 32, [0.5, 1.0, 1.75], 3, True),                      # landscape, non-square windows at the border
    (33, 33, 48, 32, [0.75, 1.5], 4, False),                          # no flip, odd size
]


def main():
    sys.path.insert(0, os.environ["LSEG_REFERENCE_ROOT"])
    with contextlib.redirect_stdout(io.StringIO()):
        import additional_utils.models as ref_models
    torch.Tensor.cuda = lambda self, *a, **k: self  # the reference hard-codes .cuda(); we are on CPU
    out = {}
    for i, (h, w, base, crop, scales, K, flip) in enumerate(CASES):
        net = StandInNet(K, crop, seed=100 + i)

        class Module(nn.Module):  # what LSeg_MultiEvalModule reads from the Lightning module
            def __init__(self):
                super().__init__()
                self.base_size, self.crop_size = base, crop
                self._up_kwargs = {"mode": "bilinear", "align_corners": True}
                self.mean, self.std = [0.5, 0.5, 0.5], [0.5, 0.5, 0.5]

            def evaluate_random(self, x, label_set):
                return net(x, label_set)

        g = torch.Generator().manual_seed(7 + i)
        image = torch.randn(1, 3, h, w, generator=g).clamp(-1, 1)
        with contextlib.redirect_stdout(io.StringIO()):
            ev = ref_models.LSeg_MultiEvalModule(Module(), device_ids=None, flip=flip, scales=scales)
            with torch.no_grad():
                scores = ev.forward(image, ["c%d" % k for k in range(K)])
        out[f"image{i}"] = image.numpy()
        out[f"scores{i}"] = scores.numpy()
        out[f"cfg{i}"] = np.array([h, w, base, crop, K, int(flip), 100 + i], dtype=np.int64)
        out[f"scales{i}"] = np.array(scales, dtype=np.float64)
    path = os.path.join(ROOT, "tests", "golden", "ref_multiscale.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, {k: v.shape for k, v in out.items() if k.startswith("scores")})


if __name__ == "__main__":
    main()

"""TEST INFRASTRUCTURE — golden fixtures that let the reference-caller tests run without the reference tree.

Runs only where a lang-seg checkout is named by LSEG_REFERENCE_ROOT:

  tests/golden/ref_live_small.npz : the UNMODIFIED reference LSegNet.forward on one 64x64 image, labels
                                    cat / other / tree (tests/test_oracle.py::test_live_reference_small)
  tests/golden/ref_callers.json   : how the reference's own Lightning module (modules/lseg_module.py,
                                    modules/lsegmentation_module.py) builds and calls its network, recorded through a
                                    stand-in LSegNet bound in place of modules.models.lseg_net: constructor keywords,
                                    the attributes it sets on the net afterwards, the attributes LSeg_MultiEvalModule
                                    reads from the module, and for forward / evaluate / evaluate_random the way the
                                    net is called (tests/test_reference_callers_gpu.py replays it around lseg_b200)

Usage:  LSEG_REFERENCE_ROOT=<lang-seg checkout> python oracle/make_golden_callers.py
"""
import json
import os
import sys
import types

import numpy as np
import torch
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import lseg_oracle as O  # noqa: E402
from oracle import ref_standins as R  # noqa: E402
from oracle import synth  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def live_small():
    sd = synth.make_state_dict(0)
    labels = ["cat", "other", "tree"]
    net = R.build_reference_net(sd, labels)
    x = synth.make_image(1, 64, 64, seed=9)
    with torch.no_grad():
        ref = net(x)
    got = O.lseg_forward(x, synth.tokenize(labels), sd)
    print(f"live small: oracle vs reference max rel err {((got - ref).abs().max() / ref.abs().max()).item():.3e}")
    np.savez_compressed(os.path.join(GOLD, "ref_live_small.npz"), logits=ref.float().numpy(),
                        labels=np.array(labels), seed=np.array(9), shape=np.array(x.shape))


class _Recorder:
    """Attribute holder that logs every assignment under its dotted path."""

    def __init__(self, path, log):
        object.__setattr__(self, "_path", path)
        object.__setattr__(self, "_log", log)

    def __getattr__(self, name):
        child = _Recorder(f"{self._path}.{name}", self._log)
        object.__setattr__(self, name, child)
        return child

    def __setattr__(self, name, value):
        self._log.append([f"{self._path}.{name}", list(value) if isinstance(value, tuple) else value])
        object.__setattr__(self, name, value)


def caller_protocol():
    R.install()
    log = {"init": None, "pokes": [], "calls": []}

    class RecordingNet(nn.Module):
        def __init__(self, labels, **kwargs):
            super().__init__()
            log["init"] = {"labels": list(labels), "kwargs": kwargs}
            self.labels = labels
            self.w = nn.Parameter(torch.zeros(1))
            self._via_call = False
            self.register_forward_pre_hook(lambda m, a: setattr(m, "_via_call", True))

        def __getattr__(self, name):
            if name == "pretrained":
                rec = _Recorder("pretrained", log["pokes"])
                self.__dict__["pretrained"] = rec
                return rec
            return super().__getattr__(name)

        def forward(self, *args, **kwargs):
            log["calls"].append({"via_call": self._via_call, "nargs": len(args), "kwargs": sorted(kwargs),
                                 "labelset_is_argument": len(args) > 1 and args[1] is _LABELS})
            self._via_call = False
            return args[0]

    shim = types.ModuleType("modules.models.lseg_net")
    shim.LSegNet = RecordingNet
    for name in ("modules.lseg_module", "modules.lsegmentation_module", "modules.models.lseg_net"):
        sys.modules.pop(name, None)
    sys.modules["modules.models.lseg_net"] = shim
    cwd = os.getcwd()
    os.chdir(R.REFERENCE_ROOT)
    try:
        from modules.lseg_module import LSegModule
        module = LSegModule(**R.MODULE_KW)
    finally:
        os.chdir(cwd)
        sys.modules.pop("modules.models.lseg_net", None)
    x = torch.zeros(1, 3, 32, 32)
    calls = {}
    for name, fn in (("forward", lambda: module(x)), ("evaluate", lambda: module.evaluate(x)),
                     ("evaluate_random", lambda: module.evaluate_random(x, _LABELS))):
        n = len(log["calls"])
        fn()
        assert len(log["calls"]) == n + 1, name
        calls[name] = log["calls"][-1]
    assert log["init"]["labels"] == synth.ade20k_labels()  # label_files/ade20k_objectInfo150.txt (tests/golden copy)
    return {
        "net_labels": "ade20k_objectInfo150",
        "net_kwargs": log["init"]["kwargs"],
        "pokes": log["pokes"],
        "module": {"base_size": module.base_size, "crop_size": module.crop_size, "mean": list(module.mean),
                   "std": list(module.std), "up_kwargs": dict(module._up_kwargs)},
        "state_dict_keys_besides_net": sorted(k for k in module.state_dict() if not k.startswith("net.")),
        "calls": calls,
    }


_LABELS = ["cat", "other", "tree", "sky"]


def main():
    torch.set_num_threads(min(16, os.cpu_count() or 1))
    live_small()
    proto = caller_protocol()
    with open(os.path.join(GOLD, "ref_callers.json"), "w") as f:
        json.dump(proto, f, indent=1, sort_keys=True)
        f.write("\n")
    print(json.dumps(proto, sort_keys=True))


if __name__ == "__main__":
    main()

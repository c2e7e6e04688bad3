"""The reference's OWN callers driving the B200 drop-in on a GPU (SURVEY.md section 8(b); the north star names exactly
these: modules/lseg_module.py, modules/lsegmentation_module.py, additional_utils/models.py).

tests/golden/ref_callers.json records, from the unmodified reference (oracle/make_golden_callers.py), how its Lightning
module builds the network (constructor keywords, the attribute it sets afterwards), what LSeg_MultiEvalModule reads
from the module, and how forward / evaluate / evaluate_random call the network. `ReferenceCaller` replays exactly that
around lseg_b200's LSegNet, so INTEGRATION.md's one-line import swap is exercised without the reference tree. The
multi-scale glue of LSeg_MultiEvalModule itself is pinned against the reference class by tests/golden/ref_multiscale.npz
(tests/test_evaluator_cpu.py, tests/test_evaluator_gpu.py).
"""
import json
import os
import threading

import pytest
import torch

from parity_util import oracle_forward, oracle_threads, rel_err, state_dict, synth
from test_model_gpu import FULL_LOGIT_REL, _report, logit_tolerance, margin_eps
from parity_util import argmax_report

pytestmark = pytest.mark.gpu
oracle_threads()

with open(os.path.join(os.path.dirname(__file__), "golden", "ref_callers.json")) as _f:
    PROTOCOL = json.load(_f)


class ReferenceCaller(torch.nn.Module):
    """LSegModule / LSegmentationModule as recorded in ref_callers.json, around lseg_b200's LSegNet."""

    def __init__(self):
        super().__init__()
        from lseg_b200 import tokenizer
        from lseg_b200.lseg_net import LSegNet
        tokenizer.enable_stand_in()  # synthetic weights, no BPE vocabulary
        assert PROTOCOL["net_labels"] == "ade20k_objectInfo150"
        self.net = LSegNet(labels=synth.ade20k_labels(), **PROTOCOL["net_kwargs"])
        for path, value in PROTOCOL["pokes"]:
            *parents, name = path.split(".")
            obj = self.net
            for p in parents:
                obj = getattr(obj, p)
            setattr(obj, name, tuple(value) if isinstance(value, list) else value)
        m = PROTOCOL["module"]
        self.base_size, self.crop_size = m["base_size"], m["crop_size"]
        self.mean, self.std, self._up_kwargs = m["mean"], m["std"], m["up_kwargs"]

    def _call(self, name, x, labelset=None):
        c = PROTOCOL["calls"][name]
        assert not c["kwargs"] and c["labelset_is_argument"] == (labelset is not None)
        args = (x, labelset)[: c["nargs"]]
        return self.net(*args) if c["via_call"] else self.net.forward(*args)

    def forward(self, x):
        return self._call("forward", x)

    def evaluate(self, x):
        return self._call("evaluate", x)

    def evaluate_random(self, x, labelset):
        return self._call("evaluate_random", x, labelset)


@pytest.fixture(scope="module")
def module():
    import lseg_b200  # noqa: F401
    m = ReferenceCaller()
    m.net.load_state_dict(state_dict(0))
    return m.cuda().eval()


def test_lsegmodule_constructs_and_pokes_img_size(module):
    # modules/lseg_module.py:86-89 pokes this attribute after construction
    assert module.net.pretrained.model.patch_embed.img_size == (480, 480)
    assert module.base_size == 520 and module.crop_size == 480
    assert len(module.net.labels) == 150


def test_evaluate_random_and_forward_match_oracle(module):
    """LSegmentationModule.evaluate_random / forward / evaluate (modules/lsegmentation_module.py:40-59)."""
    labels = ["cat", "other", "tree", "sky"]
    x = synth.make_image(2, 96, 128, seed=41)
    ref, _ = oracle_forward(x, synth.tokenize(labels))
    with torch.no_grad():
        got = module.evaluate_random(x.cuda(), labels)
    d = {"logits": rel_err(got, ref)}
    d.update(argmax_report(got, ref, margin_eps(ref)))
    _report("reference_caller_evaluate_random", d)
    assert d["logits"] <= logit_tolerance(ref, FULL_LOGIT_REL) and d["ok"], d
    ref150, _ = oracle_forward(x[:1], synth.tokenize(synth.ade20k_labels()))
    with torch.no_grad():
        a = module(x[:1].cuda())            # LightningModule.forward -> self.net(x) with the constructor's 150 labels
        b = module.evaluate(x[:1].cuda())   # -> self.net.forward(x)
    assert torch.equal(a, b)
    assert rel_err(a, ref150) <= logit_tolerance(ref150, FULL_LOGIT_REL)


def test_parent_wrapper_checkpoint_load(module):
    """Lightning checkpoints prefix every key with `net.` and carry clip_pretrained.visual.* / timm head.*; loading
    through the PARENT module with strict=True must work and must re-pack the engine weights (ADVICE r1)."""
    assert PROTOCOL["state_dict_keys_besides_net"] == []  # the reference module holds no state besides its net
    sd = synth.make_state_dict(1, with_clip_visual_stub=True)
    x = synth.make_image(1, 64, 64, seed=2).cuda()
    before = module.evaluate_random(x, ["a", "b"]).clone()
    module.load_state_dict({"net." + k: v for k, v in sd.items()}, strict=True)
    after = module.evaluate_random(x, ["a", "b"])
    assert not torch.equal(before, after), "engine kept serving the previously packed weights"
    module.load_state_dict({"net." + k: v for k, v in state_dict(0).items()}, strict=False)
    again = module.evaluate_random(x, ["a", "b"])
    assert torch.equal(before, again)


def test_multi_eval_module_threads_and_replicas(module):
    """additional_utils/models.py: LSeg_MultiEvalModule.forward (sequential multi-scale / flip / sliding window, one
    batch-1 evaluate_random per window and flip) and parallel_forward (DataParallel.replicate + one thread per GPU,
    :35-53,183-248) around the drop-in; the batched evaluator of lseg_b200 must reproduce the sequential algorithm bit
    for bit on the same network."""
    from lseg_b200.evaluator import MultiScaleEvaluator
    scales = [0.75, 1.25]
    kw = dict(base_size=module.base_size, crop_size=module.crop_size, mean=module.mean, std=module.std,
              up_kwargs=module._up_kwargs, scales=scales, flip=True)
    labels = ["cat", "other", "tree"]
    img = synth.make_image(1, 300, 400, seed=8).cuda()
    replica = torch.nn.parallel.replicate(module, [img.device.index])[0]
    par = {}

    def worker():
        with torch.no_grad():
            par["out"] = MultiScaleEvaluator(replica.evaluate_random, fused=False, max_batch=1, **kw)(img, labels)

    with torch.no_grad():
        seq = MultiScaleEvaluator(module.evaluate_random, fused=False, max_batch=1, **kw)(img, labels)
        t = threading.Thread(target=worker)
        t.start()
        t.join()
    assert seq.shape == (1, 3, 300, 400)
    assert torch.equal(seq, par["out"])
    glue = MultiScaleEvaluator(module.net, fused=False, **kw)(img, labels)
    assert torch.equal(glue, seq), f"batched evaluator differs from the sequential algorithm: {rel_err(glue, seq):.3e}"
    fused = MultiScaleEvaluator(module.net, **kw)(img, labels)
    # gather kernels instead of the torch glue: the network inputs agree to fp32 rounding (tests/test_evaluator_gpu.py), but
    # the network quantises its input to fp16, so a 1e-7 difference flips the rounding of a few hundred input pixels per crop
    assert rel_err(fused, seq) < logit_tolerance(seq, FULL_LOGIT_REL), rel_err(fused, seq)

"""CPU tests that pin the oracle (no GPU needed):
  * against the golden fixtures generated from the REAL reference (oracle/make_golden.py);
  * the restated third-party blocks (timm ViT block, CLIP text tower) against transformers' independent
    implementations with shared random weights (SURVEY.md section 8(c) item 2);
  * a small forward of the reference's own files, recorded as a fixture (oracle/make_golden_callers.py).
"""
import json
import os

import numpy as np
import pytest
import torch

from parity_util import O, rel_err, state_dict, synth

GOLD = os.path.join(os.path.dirname(__file__), "golden")
torch.set_num_threads(max(1, min(16, os.cpu_count() or 1)))

# The reference's text tower (nn.MultiheadAttention, fp16) and the restated one differ by fp16 rounding
# order only; measured 2.0e-3 of max|logit| when the fixtures were generated (make_golden.py log).
TEXT_FP16_TOL = 3e-3

# The image trunk is restated op for op: bit-identical to the fixtures on the CPU they were recorded on. Another x86
# vector ISA (the AVX2 / SSE4 kernels of MKL, oneDNN and ATen) sums fp32 in another order: measured 1.1e-6 of max|t| on
# a trunk row and 8e-6 on a tensor mean. TRUNK_REL bounds the former, TRUNK_STATS_RTOL the latter.
TRUNK_REL = 1e-5
TRUNK_STATS_RTOL = 5e-5


def assert_trunk_row(got, want):
    assert rel_err(got, torch.from_numpy(want)) <= TRUNK_REL, rel_err(got, torch.from_numpy(want))


def test_small_golden_matches_oracle():
    z = np.load(os.path.join(GOLD, "ref_small.npz"))
    labels = [str(s) for s in z["labels"]]
    x = synth.make_image(2, 64, 96, seed=2064)
    out, st = O.lseg_forward(x, synth.tokenize(labels), state_dict(0), return_stages=True)
    ref = torch.from_numpy(z["logits"])
    assert out.shape == ref.shape == (2, 5, 64, 96)
    assert rel_err(out, ref) < TEXT_FP16_TOL
    # the image trunk is restated op for op -> identical intermediate tensors up to the CPU's fp32 summation order
    assert_trunk_row(st["taps"][3][0, 0], z["tap3_row0"])
    for i in range(4):
        t = st["taps"][i]
        got = np.array([t.mean().item(), t.std().item(), t.abs().max().item()])
        assert np.allclose(got, z["taps_stats"][i], rtol=TRUNK_STATS_RTOL, atol=1e-7)


@pytest.mark.parametrize("tag,labels", [("k2", ["cat", "other"]), ("k150", None)])
def test_480_golden_matches_oracle(tag, labels):
    """BASELINE.json configs[0] (K=2) and configs[1] at B=1 (K=150), 480x480."""
    z = np.load(os.path.join(GOLD, f"ref_480_{tag}.npz"))
    labels = labels or synth.ade20k_labels()
    x = synth.make_image(1, 480, 480, seed=1480)
    out, st = O.lseg_forward(x, synth.tokenize(labels), state_dict(0), return_stages=True)
    lat = torch.from_numpy(z["logits_lattice"])
    assert rel_err(out[:, :, ::8, ::8], lat) < TEXT_FP16_TOL
    assert_trunk_row(st["taps"][3][0, 0], z["tap3_row0"])
    tf = torch.from_numpy(z["text_features"]).float()
    cos = torch.nn.functional.cosine_similarity(st["text_features"].float(), tf, dim=-1)
    assert cos.min() > 0.9999
    # masks: identical wherever the reference's own top-2 margin exceeds twice the logit tolerance
    ref_mask = torch.from_numpy(z["argmax"].astype(np.int64))
    margin = torch.from_numpy(z["margin_f16"].astype(np.float32))
    mism = out.argmax(1) != ref_mask
    eps = 2 * TEXT_FP16_TOL * float(lat.abs().max())
    assert not (mism & (margin > eps)).any(), "argmax flipped on a pixel that is not a near tie"
    if tag == "k150":
        _text_tower_reference_floor(out, st, z, tf, lat, ref_mask)


def _text_tower_reference_floor(out, st, z, tf, lat, ref_mask):
    """The floor every GPU tolerance on the text tower rests on (tests/test_model_gpu.py docstring): the reference's own
    two executions of its fp16 CLIP text tower — torch's nn.MultiheadAttention fast path inside the unmodified
    reference modules (the golden fixture) and the step-by-step multi_head_attention_forward recipe (the oracle) —
    sit ~1.7e-3 apart in the features, ~2e-3 in the logits, and disagree on ~2 % of the argmax pixels, although every
    single op agrees to the fp16 ulp (tools/text_tower_floor.py reproduces the per-op and end-to-end numbers)."""
    feat = rel_err(st["text_features"], tf)
    logit = rel_err(out[:, :, ::8, ::8], lat)
    agree = (out.argmax(1) == ref_mask).float().mean().item()
    top2 = out.topk(2, dim=1).values
    flips = out.argmax(1) != ref_mask
    quantum = 2.0 ** (int(np.floor(np.log2(float(out.abs().max())))) - 10)
    worst_quanta = float((top2[:, 0] - top2[:, 1])[flips].max()) / quantum
    print(f"reference-vs-oracle floor: text features {feat:.3e}, logits {logit:.3e}, argmax agreement {agree:.4f}, "
          f"worst flipped margin {worst_quanta:.2f} fp16 quanta")
    assert 3.0 < worst_quanta < 6.0, worst_quanta  # the GPU tests allow 6 quanta with the GPU text tower
    assert 1.0e-3 < feat < 2.5e-3, feat
    assert 1.0e-3 < logit < 3.0e-3, logit
    assert 0.97 < agree < 0.995, agree


def test_text_tower_reference_floor():
    """Alias so the floor shows up under its own name (the work is done inside the k150 golden test)."""
    z = np.load(os.path.join(GOLD, "ref_480_k150.npz"))
    tw = O.clip_text_weights_fp16(state_dict(0))
    ref = O.clip_encode_text(synth.tokenize(synth.ade20k_labels()), tw).float()
    ref = ref / ref.norm(dim=-1, keepdim=True)
    feat = rel_err(ref, torch.from_numpy(z["text_features"]).float())
    assert 1.0e-3 < feat < 2.5e-3, feat


def test_zero_shot_golden_matches_oracle():
    z = np.load(os.path.join(GOLD, "ref_zs.npz"))
    names = [line.strip() for line in open(os.path.join(GOLD, "fewshot_pascal.txt")) if line.strip()]
    texts = [synth.tokenize(["others", n]) for n in names]
    x = synth.make_image(3, 96, 96, seed=77)
    out = O.lseg_forward_zs(x, torch.from_numpy(z["class_info"]), texts, state_dict(0))
    assert rel_err(out, torch.from_numpy(z["logits"])) < TEXT_FP16_TOL


def test_head_block_golden():
    """arch_option 1 / 2: the oracle's head_block on the reference's own pre-block logits reproduces the reference module
    bit for bit (fixture generated by oracle/make_golden_arch.py from the unmodified bottleneck_block / depthwise_block)."""
    z = np.load(os.path.join(GOLD, "ref_arch.npz"))
    sd = synth.make_state_dict(0, head_block=True)
    for tag, kw in (("opt1", dict(arch_option=1, block_depth=2, activation="lrelu")),
                    ("opt2", dict(arch_option=2, block_depth=3, activation="tanh"))):
        got = O.head_block(torch.from_numpy(z[f"{tag}_pre_block"]), sd, **kw)
        assert torch.equal(got, torch.from_numpy(z[f"{tag}_post_block"]))
    # the extra keys are the only difference to the plain state dict
    base = state_dict(0)
    assert all(torch.equal(sd[k], v) for k, v in base.items())
    assert set(sd) - set(base) == {"scratch.head_block.depthwise.depthwise.weight",
                                   "scratch.head_block.depthwise.depthwise.bias"}


def test_text_tower_vs_transformers():
    """Restated CLIP encode_text (fp32 variant) vs transformers.CLIPTextModelWithProjection."""
    tr = pytest.importorskip("transformers")
    cfg = tr.CLIPTextConfig(vocab_size=49408, hidden_size=512, intermediate_size=2048, projection_dim=512,
                            num_hidden_layers=12, num_attention_heads=8, max_position_embeddings=77,
                            hidden_act="quick_gelu", layer_norm_eps=1e-5, eos_token_id=49407, bos_token_id=49406,
                            pad_token_id=0, attn_implementation="eager")
    model = tr.CLIPTextModelWithProjection(cfg).eval()
    sd = state_dict(0)
    c = "clip_pretrained."
    new = {"text_model.embeddings.token_embedding.weight": sd[c + "token_embedding.weight"],
           "text_model.embeddings.position_embedding.weight": sd[c + "positional_embedding"],
           "text_model.final_layer_norm.weight": sd[c + "ln_final.weight"],
           "text_model.final_layer_norm.bias": sd[c + "ln_final.bias"],
           "text_projection.weight": sd[c + "text_projection"].t().contiguous()}
    for i in range(12):
        s, d = f"{c}transformer.resblocks.{i}.", f"text_model.encoder.layers.{i}."
        wq, wk, wv = sd[s + "attn.in_proj_weight"].chunk(3, 0)
        bq, bk, bv = sd[s + "attn.in_proj_bias"].chunk(3, 0)
        for n, w_, b_ in (("q_proj", wq, bq), ("k_proj", wk, bk), ("v_proj", wv, bv)):
            new[d + f"self_attn.{n}.weight"], new[d + f"self_attn.{n}.bias"] = w_, b_
        new[d + "self_attn.out_proj.weight"] = sd[s + "attn.out_proj.weight"]
        new[d + "self_attn.out_proj.bias"] = sd[s + "attn.out_proj.bias"]
        for a, b in (("layer_norm1", "ln_1"), ("layer_norm2", "ln_2")):
            new[d + a + ".weight"], new[d + a + ".bias"] = sd[s + b + ".weight"], sd[s + b + ".bias"]
        for a, b in (("mlp.fc1", "mlp.c_fc"), ("mlp.fc2", "mlp.c_proj")):
            new[d + a + ".weight"], new[d + a + ".bias"] = sd[s + b + ".weight"], sd[s + b + ".bias"]
    missing, unexpected = model.load_state_dict(new, strict=False)
    assert not unexpected and all("position_ids" in m for m in missing), (missing, unexpected)
    tokens = synth.tokenize(["wall", "traffic light", "chest of drawers", "a photo of a very small cat"])
    with torch.no_grad():
        ref = model(input_ids=tokens, attention_mask=None).text_embeds
    tw = O.clip_text_weights_fp16(sd, dtype=torch.float32)
    got = O.clip_encode_text(tokens, tw, dtype=torch.float32)
    assert rel_err(got, ref) < 2e-5


def test_vit_block_vs_transformers():
    """Restated timm Block vs transformers.ViTLayer with shared weights (exact-erf GELU, LN eps 1e-6)."""
    tr = pytest.importorskip("transformers")
    from transformers.models.vit.modeling_vit import ViTLayer
    cfg = tr.ViTConfig(hidden_size=1024, num_attention_heads=16, intermediate_size=4096, hidden_act="gelu",
                       layer_norm_eps=1e-6, qkv_bias=True, attn_implementation="eager",
                       hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    layer = ViTLayer(cfg).eval()
    sd = state_dict(0)
    p = "pretrained.model.blocks.7."
    wq, wk, wv = sd[p + "attn.qkv.weight"].chunk(3, 0)
    bq, bk, bv = sd[p + "attn.qkv.bias"].chunk(3, 0)
    new = {"attention.attention.query.weight": wq, "attention.attention.query.bias": bq,
           "attention.attention.key.weight": wk, "attention.attention.key.bias": bk,
           "attention.attention.value.weight": wv, "attention.attention.value.bias": bv,
           "attention.output.dense.weight": sd[p + "attn.proj.weight"],
           "attention.output.dense.bias": sd[p + "attn.proj.bias"],
           "layernorm_before.weight": sd[p + "norm1.weight"], "layernorm_before.bias": sd[p + "norm1.bias"],
           "layernorm_after.weight": sd[p + "norm2.weight"], "layernorm_after.bias": sd[p + "norm2.bias"],
           "intermediate.dense.weight": sd[p + "mlp.fc1.weight"], "intermediate.dense.bias": sd[p + "mlp.fc1.bias"],
           "output.dense.weight": sd[p + "mlp.fc2.weight"], "output.dense.bias": sd[p + "mlp.fc2.bias"]}
    layer.load_state_dict(new, strict=True)
    x = torch.randn(2, 37, 1024, generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        ref = layer(x)
        ref = ref[0] if isinstance(ref, (tuple, list)) else ref
        got = O.vit_block(x, sd, p)
    assert rel_err(got, ref) < 2e-5


def test_attention_hook_corroboration():
    """In-tree corroboration of the restated attention: lseg_vit.py:22-42's get_attention hook recomputes
    softmax(q k^T * scale) from module.qkv; the oracle's attention weights must be that same formula."""
    sd = state_dict(0)
    p = "pretrained.model.blocks.0.attn."
    x = torch.randn(1, 17, 1024, generator=torch.Generator().manual_seed(1))
    qkv = torch.nn.functional.linear(x, sd[p + "qkv.weight"], sd[p + "qkv.bias"]).reshape(1, 17, 3, 16, 64)
    q, k, v = qkv.permute(2, 0, 3, 1, 4)
    attn = ((q @ k.transpose(-2, -1)) * 64 ** -0.5).softmax(dim=-1)
    out = (attn @ v).transpose(1, 2).reshape(1, 17, 1024)
    out = torch.nn.functional.linear(out, sd[p + "proj.weight"], sd[p + "proj.bias"])
    assert torch.allclose(out, O.vit_attention(x, sd, p), atol=1e-6)


def test_reference_key_contract():
    """The drop-in module carries exactly the reference's state-dict keys/shapes (SURVEY.md Appendix C)."""
    import lseg_b200  # noqa: F401
    from lseg_b200.lseg_net import LSegNet
    from parity_util import NET_KW
    want = json.load(open(os.path.join(GOLD, "state_dict_keys.json")))
    net = LSegNet(labels=["a", "b"], **NET_KW)
    have = {k: list(v.shape) for k, v in net.state_dict().items()}
    assert have == want
    # and accepts real-checkpoint extras (unused CLIP visual tower, timm classifier head)
    sd = dict(state_dict(0))
    sd["clip_pretrained.visual.conv1.weight"] = torch.zeros(4, 3, 32, 32)
    sd["pretrained.model.head.weight"] = torch.zeros(1000, 1024)
    net.load_state_dict(sd)
    assert net.text.shape == (2, 77) and net.text.dtype == torch.int64
    assert abs(float(net.logit_scale) - 14.2857) < 1e-3


@pytest.mark.parametrize("tag,backbone,layer_shapes", [
    ("b32", "clip_vitb32_384", [(96, 16, 24), (192, 8, 12), (384, 4, 6), (768, 2, 3)]),
    ("rn50x16", "clipRN50x16_vitl16_384", [(256, 16, 24), (512, 8, 12), (1024, 4, 6), (1024, 2, 3)])])
def test_other_backbone_golden_and_key_contract(tag, backbone, layer_shapes):
    """The oracle against the unmodified reference's output with that backbone (oracle/make_golden_backbones.py), trunk
    statistics to the CPU's fp32 summation order (TRUNK_STATS_RTOL), and the drop-in module's state-dict keys/shapes against the reference module's."""
    import lseg_b200  # noqa: F401
    from lseg_b200.lseg_net import LSegNet
    from parity_util import NET_KW
    z = np.load(os.path.join(GOLD, f"ref_{tag}.npz"))
    labels = [str(s) for s in z["small_labels"]]
    x = synth.make_image(2, 64, 96, seed=2064)
    sd = state_dict(0, backbone)
    out, st = O.lseg_forward(x, synth.tokenize(labels), sd, return_stages=True, backbone=backbone)
    ref = torch.from_numpy(z["small_logits"])
    assert out.shape == ref.shape == (2, 5, 64, 96)
    assert rel_err(out, ref) < 5e-3  # two executions of the fp16 text tower (measured 3.0e-3 at max|logit| ~ 0.3)
    assert_trunk_row(st["taps"][3][0, 0], z["small_tap3_row0"])
    for i in range(4):
        for name, t in (("taps", st["taps"][i]), ("layers", st["layers"][i])):
            got = np.array([t.mean().item(), t.std().item(), t.abs().max().item()])
            assert np.allclose(got, z[f"small_{name}_stats"][i], rtol=TRUNK_STATS_RTOL, atol=1e-7), (name, i)
    assert [tuple(l.shape[1:]) for l in st["layers"]] == layer_shapes
    want = json.load(open(os.path.join(GOLD, f"state_dict_keys_{tag}.json")))
    net = LSegNet(labels=["a", "b"], **{**NET_KW, "backbone": backbone})
    assert {k: list(v.shape) for k, v in net.state_dict().items()} == want
    net.load_state_dict(sd)
    assert net.out_c == st["text_features"].shape[1]
    with pytest.raises(AssertionError):  # lseg_blocks.py:53-55 failure mode for backbones that are not built
        LSegNet(labels=["a"], **{**NET_KW, "backbone": "clip_resnet101"})


def test_rn101_zero_shot_golden_and_key_contract():
    """LSegRNNetZS (ResNet-101 trunk, lseg_net_zs.py:240-378): the oracle against the unmodified reference's output
    (oracle/make_golden_rn.py), stage statistics to TRUNK_STATS_RTOL, and the drop-in module's state-dict keys/shapes."""
    import lseg_b200  # noqa: F401
    from lseg_b200.lseg_net import LSegNetZS, LSegRNNetZS
    z = np.load(os.path.join(GOLD, "ref_rn101.npz"))
    names = [line.strip() for line in open(os.path.join(GOLD, "fewshot_pascal.txt")) if line.strip()]
    texts = [synth.tokenize(["others", n]) for n in names]
    sd = state_dict(0, "clip_resnet101")
    x = synth.make_image(3, 96, 128, seed=77)
    out, st = O.lseg_forward_rn_zs(x, torch.from_numpy(z["small_class_info"]), texts, sd, return_stages=True)
    ref = torch.from_numpy(z["small_logits"])
    assert out.shape == ref.shape == (3, 2, 96, 128)
    assert rel_err(out, ref) < 1.5 * float(z["small_floor"]) + 1e-3  # two executions of the fp16 text tower
    assert [tuple(l.shape[1:]) for l in st["layers"]] == [(256, 24, 32), (512, 12, 16), (1024, 6, 8), (2048, 3, 4)]
    for k in range(4):
        t = st["layers"][k]
        got = np.array([t.mean().item(), t.std().item(), t.abs().max().item()])
        assert np.allclose(got, z["small_layers_stats"][k], rtol=TRUNK_STATS_RTOL, atol=1e-7), k
    want = json.load(open(os.path.join(GOLD, "state_dict_keys_rn101.json")))
    net = LSegRNNetZS(label_list=names, features=256, arch_option=0, block_depth=0, activation="lrelu")
    assert {k: list(v.shape) for k, v in net.state_dict().items()} == want
    net.load_state_dict(sd)
    assert net.backbone == "clip_resnet101" and len(net.texts) == len(names) and net.texts[0].shape == (2, 77)
    with pytest.raises(ValueError):  # the two zero-shot classes keep their trunks apart, like the reference's
        LSegNetZS(label_list=names, backbone="clip_resnet101", features=256, arch_option=0, block_depth=0, activation="lrelu")
    with pytest.raises(ValueError):
        LSegRNNetZS(label_list=names, backbone="clip_vitl16_384", features=256, arch_option=0, block_depth=0,
                    activation="lrelu")


def test_checkpoint_load_through_parent_module():
    """Lightning's load_from_checkpoint loads `net.`-prefixed keys on the PARENT module; torch then recurses with
    _load_from_state_dict and never calls a child's load_state_dict override. strict=True must still accept real-checkpoint
    extras and the packed weights must be invalidated (hooks on the net, not an override)."""
    import lseg_b200  # noqa: F401
    from lseg_b200.lseg_net import LSegNet
    from parity_util import NET_KW

    class Parent(torch.nn.Module):
        def __init__(self, net):
            super().__init__()
            self.net = net

    net = LSegNet(labels=["a", "b"], **NET_KW)
    parent = Parent(net)
    net._shared["text_cache"]["sentinel"] = 1
    sd = {"net." + k: v for k, v in synth.make_state_dict(0, with_clip_visual_stub=True).items()}
    sd["net.pretrained.model.head.weight"] = torch.zeros(1000, 1024)
    res = parent.load_state_dict(sd, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    assert "sentinel" not in net._shared["text_cache"], "load through the parent did not invalidate the engine state"
    assert torch.equal(net.scratch.head1.bias, sd["net.scratch.head1.bias"])


def test_tokenizer_contract():
    import lseg_b200  # noqa: F401
    from lseg_b200.tokenizer import tokenize
    labels = synth.ade20k_labels()
    assert len(labels) == 150 and labels[0] == "wall" and labels[1] == "building"
    a, b = tokenize(labels), synth.tokenize(labels)
    assert torch.equal(a, b) and a.dtype == torch.int64 and a.shape == (150, 77)
    assert (a[:, 0] == 49406).all() and (a.max(dim=1).values == 49407).all()
    with pytest.raises(RuntimeError):
        tokenize(["w " * 100])


def test_live_reference_small():
    """The unmodified reference LSegNet.forward on one 64x64 image, as recorded by oracle/make_golden_callers.py."""
    z = np.load(os.path.join(GOLD, "ref_live_small.npz"))
    labels = [str(s) for s in z["labels"]]
    x = synth.make_image(*[int(v) for v in z["shape"][[0, 2, 3]]], seed=int(z["seed"]))
    ref = torch.from_numpy(z["logits"])
    got = O.lseg_forward(x, synth.tokenize(labels), state_dict(0))
    assert got.shape == ref.shape == (1, 3, 64, 64)
    assert rel_err(got, ref) < TEXT_FP16_TOL

"""TEST INFRASTRUCTURE — stand-ins that let the reference's own modules import and run unchanged.

The reference depends on third-party packages that are not installed here (timm 0.4.12, OpenAI clip
@04f4dc2, PyTorch-Encoding, pytorch_lightning, matplotlib; SURVEY.md Appendix B). This module registers
`sys.modules` stand-ins for them:
  * `timm.create_model("vit_large_patch16_384")`  -> a faithful nn.Module restatement of the timm 0.4.12
    VisionTransformer (attribute and parameter names as the reference touches them, Appendix A.1);
  * `clip.load("ViT-B/32")` -> the CLIP text tower as nn.Modules (nn.MultiheadAttention, QuickGELU,
    fp32-computing LayerNorm), weights converted to fp16 like clip.load(device='cuda') does;
    `clip.tokenize` -> oracle.synth.tokenize (no BPE vocabulary offline);
  * inert stubs for encoding / pytorch_lightning / matplotlib so modules/lseg_module.py imports.
Used by the fixture generators oracle/make_golden*.py and by bench.py --impl reference (which falls back to the oracle
restatement when no reference checkout is given); nothing here is imported by the product path. The checkout is named
by the environment variable LSEG_REFERENCE_ROOT.
"""
import os
import sys
import types
from collections import OrderedDict

import torch
import torch.nn as nn

REFERENCE_ROOT = os.environ.get("LSEG_REFERENCE_ROOT", "")  # a lang-seg checkout


def reference_available():
    return bool(REFERENCE_ROOT) and os.path.isdir(os.path.join(REFERENCE_ROOT, "modules", "models"))


# ---------------------------------------------------------------------------------------------
# timm 0.4.12 VisionTransformer (Appendix A.1)
# ---------------------------------------------------------------------------------------------
class _Mlp(nn.Module):
    def __init__(self, dim, hidden):
        super().__init__()
        self.fc1 = nn.Linear(dim, hidden)
        self.act = nn.GELU()
        self.fc2 = nn.Linear(hidden, dim)
        self.drop = nn.Dropout(0.0)

    def forward(self, x):
        return self.drop(self.fc2(self.drop(self.act(self.fc1(x)))))


class _Attention(nn.Module):
    def __init__(self, dim, num_heads):
        super().__init__()
        self.num_heads = num_heads
        self.scale = (dim // num_heads) ** -0.5
        self.qkv = nn.Linear(dim, dim * 3, bias=True)
        self.attn_drop = nn.Dropout(0.0)
        self.proj = nn.Linear(dim, dim)
        self.proj_drop = nn.Dropout(0.0)

    def forward(self, x):
        B, N, C = x.shape
        qkv = self.qkv(x).reshape(B, N, 3, self.num_heads, C // self.num_heads).permute(2, 0, 3, 1, 4)
        q, k, v = qkv[0], qkv[1], qkv[2]
        attn = (q @ k.transpose(-2, -1)) * self.scale
        attn = self.attn_drop(attn.softmax(dim=-1))
        x = (attn @ v).transpose(1, 2).reshape(B, N, C)
        return self.proj_drop(self.proj(x))


class _Block(nn.Module):
    def __init__(self, dim, num_heads, mlp_ratio=4.0):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim, eps=1e-6)
        self.attn = _Attention(dim, num_heads)
        self.drop_path = nn.Identity()
        self.norm2 = nn.LayerNorm(dim, eps=1e-6)
        self.mlp = _Mlp(dim, int(dim * mlp_ratio))

    def forward(self, x):
        x = x + self.drop_path(self.attn(self.norm1(x)))
        x = x + self.drop_path(self.mlp(self.norm2(x)))
        return x


class _PatchEmbed(nn.Module):
    def __init__(self, img_size, patch, in_chans, dim):
        super().__init__()
        self.img_size = (img_size, img_size)
        self.patch_size = (patch, patch)
        self.proj = nn.Conv2d(in_chans, dim, kernel_size=patch, stride=patch)


class VisionTransformer(nn.Module):
    def __init__(self, img_size=384, patch=16, dim=1024, depth=24, heads=16):
        super().__init__()
        self.patch_embed = _PatchEmbed(img_size, patch, 3, dim)
        n = (img_size // patch) ** 2
        self.cls_token = nn.Parameter(torch.zeros(1, 1, dim))
        self.pos_embed = nn.Parameter(torch.zeros(1, n + 1, dim))
        self.pos_drop = nn.Dropout(0.0)
        self.blocks = nn.ModuleList([_Block(dim, heads) for _ in range(depth)])
        self.norm = nn.LayerNorm(dim, eps=1e-6)
        self.pre_logits = nn.Identity()


def _timm_create_model(name, pretrained=False, **kw):
    if name == "vit_large_patch16_384":
        return VisionTransformer()
    if name == "vit_base_patch32_384":  # timm 0.4.12 vision_transformer.py: patch 32, dim 768, depth 12, 12 heads
        return VisionTransformer(patch=32, dim=768, depth=12, heads=12)
    raise NotImplementedError(name)


# ---------------------------------------------------------------------------------------------
# CLIP @04f4dc2 text tower (Appendix A.2)
# ---------------------------------------------------------------------------------------------
class _ClipLayerNorm(nn.LayerNorm):
    def forward(self, x):
        orig = x.dtype
        ret = torch.nn.functional.layer_norm(x.float(), self.normalized_shape, self.weight.float(),
                                             self.bias.float(), self.eps)
        return ret.type(orig)


class _QuickGELU(nn.Module):
    def forward(self, x):
        return x * torch.sigmoid(1.702 * x)


class _ResidualAttentionBlock(nn.Module):
    def __init__(self, d_model, n_head, attn_mask):
        super().__init__()
        self.attn = nn.MultiheadAttention(d_model, n_head)
        self.ln_1 = _ClipLayerNorm(d_model)
        self.mlp = nn.Sequential(OrderedDict([("c_fc", nn.Linear(d_model, d_model * 4)), ("gelu", _QuickGELU()),
                                              ("c_proj", nn.Linear(d_model * 4, d_model))]))
        self.ln_2 = _ClipLayerNorm(d_model)
        self.attn_mask = attn_mask

    def attention(self, x):
        mask = self.attn_mask.to(dtype=x.dtype, device=x.device)
        return self.attn(x, x, x, need_weights=False, attn_mask=mask)[0]

    def forward(self, x):
        x = x + self.attention(self.ln_1(x))
        x = x + self.mlp(self.ln_2(x))
        return x


class _Transformer(nn.Module):
    def __init__(self, width, layers, heads, attn_mask):
        super().__init__()
        self.resblocks = nn.Sequential(*[_ResidualAttentionBlock(width, heads, attn_mask) for _ in range(layers)])

    def forward(self, x):
        return self.resblocks(x)


class ClipTextOnly(nn.Module):
    """CLIP with only the members LSeg touches (encode_text); the visual tower is never called."""

    def __init__(self, embed_dim=512, context_length=77, vocab_size=49408, width=512, heads=8, layers=12):
        super().__init__()
        self.context_length = context_length
        mask = torch.empty(context_length, context_length).fill_(float("-inf")).triu_(1)
        self.transformer = _Transformer(width, layers, heads, mask)
        self.token_embedding = nn.Embedding(vocab_size, width)
        self.positional_embedding = nn.Parameter(torch.empty(context_length, width))
        self.ln_final = _ClipLayerNorm(width)
        self.text_projection = nn.Parameter(torch.empty(width, embed_dim))
        self.logit_scale = nn.Parameter(torch.ones([]))

    @property
    def dtype(self):
        return self.transformer.resblocks[0].mlp.c_fc.weight.dtype

    def encode_text(self, text):
        x = self.token_embedding(text).type(self.dtype)
        x = x + self.positional_embedding.type(self.dtype)
        x = x.permute(1, 0, 2)
        x = self.transformer(x)
        x = x.permute(1, 0, 2)
        x = self.ln_final(x).type(self.dtype)
        return x[torch.arange(x.shape[0]), text.argmax(dim=-1)] @ self.text_projection


def _convert_weights(model):
    """clip.model.convert_weights: fp16 for Linear / MultiheadAttention params and text_projection."""
    def _to_fp16(l):
        if isinstance(l, (nn.Conv1d, nn.Conv2d, nn.Linear)):
            l.weight.data = l.weight.data.half()
            if l.bias is not None:
                l.bias.data = l.bias.data.half()
        if isinstance(l, nn.MultiheadAttention):
            for attr in ["in_proj_weight", "q_proj_weight", "k_proj_weight", "v_proj_weight", "in_proj_bias",
                         "bias_k", "bias_v"]:
                t = getattr(l, attr, None)
                if t is not None:
                    t.data = t.data.half()
        for name in ["text_projection", "proj"]:
            if hasattr(l, name):
                attr = getattr(l, name)
                if attr is not None:
                    attr.data = attr.data.half()
    model.apply(_to_fp16)


def _clip_load(name, device="cpu", jit=False):
    if name == "ViT-B/32":
        model = ClipTextOnly()
    elif name == "RN50x16":  # CLIP model card: embed_dim 768, transformer_width 768, 12 heads, 12 layers
        model = ClipTextOnly(embed_dim=768, width=768, heads=12)
    else:
        raise NotImplementedError(name)
    _convert_weights(model)  # what clip.load(device='cuda') leaves behind (lseg_vit.py:224)
    return model.eval(), None


def install(with_lightning_stack=True):
    """Register the stand-ins and put the reference checkout on sys.path. Idempotent."""
    if not reference_available():
        raise FileNotFoundError(f"no lang-seg checkout at LSEG_REFERENCE_ROOT={REFERENCE_ROOT!r}")
    here = os.path.dirname(os.path.abspath(__file__))
    sys.path.insert(0, os.path.dirname(here))
    from oracle import synth

    timm = types.ModuleType("timm")
    timm.create_model = _timm_create_model
    sys.modules["timm"] = timm

    clip = types.ModuleType("clip")
    clip.load = _clip_load
    clip.tokenize = synth.tokenize
    sys.modules["clip"] = clip

    if with_lightning_stack:
        def _mod(name, **attrs):
            m = types.ModuleType(name)
            m.__dict__.update(attrs)
            sys.modules[name] = m
            return m

        class _Dataset:
            num_class = 150

            def __init__(self, *a, **k):
                pass

            def __len__(self):
                return 0

        class _Anything:
            def __init__(self, *a, **k):
                pass

            def __call__(self, *a, **k):
                return None

        up_kwargs = {"mode": "bilinear", "align_corners": True}
        _mod("encoding")
        _mod("encoding.models", get_segmentation_model=lambda *a, **k: None)
        _mod("encoding.models.sseg", BaseNet=nn.Module)
        _mod("encoding.models.sseg.base", up_kwargs=up_kwargs)
        _mod("encoding.nn", SegmentationLosses=_Anything, SyncBatchNorm=nn.BatchNorm2d)
        _mod("encoding.utils", batch_pix_accuracy=lambda *a, **k: (0, 0),
             batch_intersection_union=lambda *a, **k: (0, 0), SegmentationMetric=_Anything)
        _mod("encoding.utils.metrics")
        _mod("encoding.datasets", get_dataset=lambda *a, **k: _Dataset(), test_batchify_fn=None,
             datasets={"ade20k": _Dataset})
        _mod("encoding.parallel", DataParallelModel=nn.DataParallel, DataParallelCriterion=nn.DataParallel)
        pl = _mod("pytorch_lightning", LightningModule=nn.Module)
        metrics = _mod("pytorch_lightning.metrics", Accuracy=_Anything)
        pl.metrics = metrics
        _mod("matplotlib")
        _mod("matplotlib.pyplot")
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)


def build_reference_net(state_dict, labels, arch_option=0, block_depth=0, activation="lrelu", backbone="clip_vitl16_384"):
    """Construct the UNMODIFIED reference LSegNet (modules/models/lseg_net.py:208-226) on CPU and load `state_dict`."""
    install()
    cwd = os.getcwd()
    os.chdir(REFERENCE_ROOT)
    try:
        from modules.models.lseg_net import LSegNet
        net = LSegNet(labels=labels, backbone=backbone, features=256, crop_size=480, arch_option=arch_option,
                      block_depth=block_depth, activation=activation)
    finally:
        os.chdir(cwd)
    missing, unexpected = net.load_state_dict(state_dict, strict=False)
    missing = [k for k in missing if "num_batches_tracked" not in k]
    assert not missing, f"state dict misses reference keys: {missing[:5]}"
    assert all(k.startswith("clip_pretrained.visual.") for k in unexpected), unexpected[:5]
    return net.eval()


MODULE_KW = dict(data_path="", dataset="ade20k", batch_size=1, base_lr=0, max_epochs=0, backbone="clip_vitl16_384",
                 num_features=256, aux=False, aux_weight=0, se_loss=False, se_weight=0, ignore_index=255, dropout=0.0,
                 scale_inv=False, augment=False, no_batchnorm=False, widehead=False, widehead_hr=False, arch_option=0,
                 block_depth=0, activation="lrelu")  # the keyword set of test_lseg.py:221-246


def build_reference_module(state_dict=None, drop_in=False, **overrides):
    """Construct the UNMODIFIED reference `LSegModule` (modules/lseg_module.py) the way test_lseg.py:221-246 does.

    drop_in=False: with the reference's own `LSegNet` (modules/models/lseg_net.py) — the CPU baseline.
    drop_in=True : the one-line import swap of INTEGRATION.md applied WITHOUT editing the file: the module name
                   `modules.models.lseg_net` is pre-bound to a shim whose `LSegNet` is lseg_b200's, so
                   `from .models.lseg_net import LSegNet` (modules/lseg_module.py:8) resolves to the B200 drop-in.
    The label file is opened relative to the cwd (modules/lseg_module.py:99), hence the chdir."""
    install()
    for name in ("modules.lseg_module", "modules.lsegmentation_module", "modules.models.lseg_net"):
        sys.modules.pop(name, None)
    if drop_in:
        import importlib
        importlib.import_module("lang-seg_b200.tokenizer").enable_stand_in()  # synthetic weights, no BPE vocabulary
        ours = importlib.import_module("lang-seg_b200.lseg_net")
        shim = types.ModuleType("modules.models.lseg_net")
        shim.LSegNet = ours.LSegNet
        sys.modules["modules.models.lseg_net"] = shim
    kw = dict(MODULE_KW)
    kw.update(overrides)
    cwd = os.getcwd()
    os.chdir(REFERENCE_ROOT)
    try:
        from modules.lseg_module import LSegModule
        module = LSegModule(**kw)
    finally:
        os.chdir(cwd)
        sys.modules.pop("modules.models.lseg_net", None) if drop_in else None
    if state_dict is not None:
        missing, unexpected = module.net.load_state_dict(state_dict, strict=False)
        missing = [k for k in missing if "num_batches_tracked" not in k]
        assert not missing, f"state dict misses keys: {missing[:5]}"
    return module.eval()


def load_multi_eval_module():
    """The unmodified `LSeg_MultiEvalModule` class (additional_utils/models.py)."""
    install()
    from additional_utils.models import LSeg_MultiEvalModule
    return LSeg_MultiEvalModule

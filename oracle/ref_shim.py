"""TEST INFRASTRUCTURE ONLY -- import the UNMODIFIED reference modules from /root/reference on CPU.

The reference pins transformers 4.30 / timm / xformers / diffusers, none of which match this image.  This
module registers ~40 lines of stub modules and back-fills three removed transformers helpers so that
`models.seed_qformer.qformer_quantizer` and `models.llama_xformer` import and run as shipped (recipe and
probes: SURVEY.md section 8c).  It exists only in the build container (the GPU box has no /root/reference);
it is used by oracle/make_golden.py to generate tests/golden/*, which the tests compare against.

Nothing here is arithmetic: the stubs replace (a) timm init helpers (trunc_normal_, to_2tuple, DropPath),
(b) three network-touching factories (BertTokenizer / BertLMHeadModel.from_pretrained / eva_vit_g.pth
download), (c) xformers.ops.memory_efficient_attention by torch SDPA (the only reference arithmetic that
lives in an un-vendored dependency: xformers >= 0.0.20, requirements.txt:4; its published semantics are
softmax(q k^T / sqrt(d) + bias) v).
"""
from __future__ import annotations

import importlib
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("SEED_REFERENCE_ROOT", "/root/reference")


def available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "models", "seed_qformer"))


_installed = False


def _install_stubs() -> None:
    global _installed
    if _installed:
        return
    import torch
    import torch.nn as nn
    import torch.nn.functional as F
    import transformers  # noqa: F401  (must be imported before the back-fill below)
    import transformers.modeling_utils as mu
    import transformers.pytorch_utils as pu

    # ---- timm (init-time helpers only; no inference arithmetic) ----
    def to_2tuple(x):
        return tuple(x) if isinstance(x, (tuple, list)) else (x, x)

    def drop_path(x, drop_prob: float = 0.0, training: bool = False):
        if drop_prob == 0.0 or not training:
            return x
        raise NotImplementedError("drop_path is training-only")

    class DropPath(nn.Module):
        def __init__(self, drop_prob=None):
            super().__init__()
            self.drop_prob = drop_prob

        def forward(self, x):
            return drop_path(x, self.drop_prob, self.training)

    class _PatchEmbed(nn.Module):  # only referenced by the unused timm-style VisionTransformer in vit.py
        def __init__(self, *a, **k):
            super().__init__()
            raise NotImplementedError

    def _mk(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    timm = _mk("timm")
    timm.models = _mk("timm.models")
    timm.models.layers = _mk("timm.models.layers", drop_path=drop_path, to_2tuple=to_2tuple,
                             trunc_normal_=nn.init.trunc_normal_, DropPath=DropPath)
    timm.models.hub = _mk("timm.models.hub", download_cached_file=lambda *a, **k: (_ for _ in ()).throw(
        RuntimeError("no network")))
    timm.models.vision_transformer = _mk("timm.models.vision_transformer", _cfg=lambda **k: k, PatchEmbed=_PatchEmbed)
    timm.models.registry = _mk("timm.models.registry", register_model=lambda f: f)
    timm.models.helpers = _mk("timm.models.helpers", named_apply=None, adapt_input_conv=None)

    # ---- transformers 4.30 helpers that moved / disappeared ----
    for name in ("apply_chunking_to_forward", "prune_linear_layer"):
        if not hasattr(mu, name):
            setattr(mu, name, getattr(pu, name))
    if not hasattr(mu, "find_pruneable_heads_and_indices"):
        mu.find_pruneable_heads_and_indices = getattr(pu, "find_pruneable_heads_and_indices", lambda *a, **k: None)

    # ---- xformers.ops (un-vendored dependency; published semantics restated with SDPA) ----
    class LowerTriangularMask:
        pass

    def memory_efficient_attention(q, k, v, attn_bias=None, p: float = 0.0, scale=None):
        # inputs [B, M, H, K]; LowerTriangularMask == causal, top-left aligned as in xformers 0.0.20
        qh, kh, vh = (t.transpose(1, 2) for t in (q, k, v))
        mask = None
        if isinstance(attn_bias, LowerTriangularMask) or attn_bias is LowerTriangularMask:
            mq, mk = qh.shape[-2], kh.shape[-2]
            mask = torch.ones(mq, mk, dtype=torch.bool, device=q.device).tril()
        elif attn_bias is not None:
            mask = attn_bias
        o = F.scaled_dot_product_attention(qh, kh, vh, attn_mask=mask, scale=scale)
        return o.transpose(1, 2)

    xf = _mk("xformers")
    xf.ops = _mk("xformers.ops", memory_efficient_attention=memory_efficient_attention,
                 LowerTriangularMask=LowerTriangularMask)
    _installed = True


def _import_reference(modname: str):
    """import `models.<modname>` from /root/reference without shadowing this repo's own `models` package."""
    if not available():
        raise RuntimeError(f"reference not found at {REFERENCE_ROOT}")
    _install_stubs()
    key = "seed_reference_models"
    if key not in sys.modules:
        pkg = types.ModuleType(key)
        pkg.__path__ = [os.path.join(REFERENCE_ROOT, "models")]
        sys.modules[key] = pkg
    return importlib.import_module(f"{key}.{modname}")


def load_quantizer_module():
    """-> the reference module models/seed_qformer/qformer_quantizer.py with network factories replaced."""
    import torch
    import torch.nn as nn

    qc = _import_reference("seed_qformer.qformer_causual")
    # transformers-5 API drift (no arithmetic): init_weights / get_head_mask
    qc.BertPreTrainedModel.init_weights = lambda self: self.apply(self._init_weights)
    qc.BertModel.get_head_mask = lambda self, head_mask, n, *a, **k: [None] * n
    blip2 = _import_reference("seed_qformer.blip2")
    eva = _import_reference("seed_qformer.eva_vit")
    qq = _import_reference("seed_qformer.qformer_quantizer")

    def init_tokenizer(cls, truncation_side="right"):
        return None  # BertTokenizer download; never used on the encode path

    def init_Qformer(cls, num_query_token, vision_width, cross_attention_freq=2):
        cfg = qc.BertConfig()  # defaults == bert-base-uncased (blip2.py:54)
        cfg.encoder_width = vision_width
        cfg.add_cross_attention = True
        cfg.cross_attention_freq = cross_attention_freq
        cfg.query_length = num_query_token
        depth = int(os.environ.get("SEED_ORACLE_QFORMER_LAYERS", cfg.num_hidden_layers))
        cfg.num_hidden_layers = depth
        model = qc.BertLMHeadModel(cfg)
        query_tokens = nn.Parameter(torch.zeros(1, num_query_token, cfg.hidden_size))
        query_tokens.data.normal_(mean=0.0, std=cfg.initializer_range)
        return model, query_tokens

    def create_eva_vit_g(img_size=224, drop_path_rate=0.4, use_checkpoint=False, precision="fp16"):
        from functools import partial
        depth = int(os.environ.get("SEED_ORACLE_VIT_DEPTH", 39))
        return eva.VisionTransformer(img_size=img_size, patch_size=14, use_mean_pooling=False, embed_dim=1408,
                                     depth=depth, num_heads=1408 // 88, mlp_ratio=4.3637, qkv_bias=True,
                                     drop_path_rate=0.0, norm_layer=partial(nn.LayerNorm, eps=1e-6),
                                     use_checkpoint=use_checkpoint)   # args of eva_vit.py:462-474, no download

    blip2.Blip2Base.init_tokenizer = classmethod(init_tokenizer)
    blip2.Blip2Base.init_Qformer = classmethod(init_Qformer)
    blip2.create_eva_vit_g = create_eva_vit_g
    return qq


def build_reference_quantizer(vit_depth: int = 39, qformer_layers: int = 12, decode_depth: int = 4):
    """Construct the reference Blip2QformerQuantizer (fp32, CPU) at a possibly reduced depth."""
    os.environ["SEED_ORACLE_VIT_DEPTH"] = str(vit_depth)
    os.environ["SEED_ORACLE_QFORMER_LAYERS"] = str(qformer_layers)
    qq = load_quantizer_module()
    model = qq.Blip2QformerQuantizer(vit_precision="fp32", decode_depth=decode_depth)
    return model.eval()


def load_llama_module():
    return _import_reference("llama_xformer")

"""Parameter containers with the reference's module / parameter names, backed by the native engine.

The classes mirror clip/model.py of the reference (same constructor signatures, attribute and
state-dict key names, so checkpoints and the freeze-by-substring rule of trainers/mudpt.py:205-212
keep working) but hold *no* PyTorch compute: `VisionTransformer_MuDPT.forward` and the text path
(trainers/mudpt.py) run the towers through libmudpt_b200.so.  nn.MultiheadAttention / nn.Linear /
nn.LayerNorm appear only as containers that own tensors with the right names and shapes.

  LayerNorm, QuickGELU ................ clip/model.py:164-175
  ResidualAttentionBlock_MuDPT ........ clip/model.py:254-301
  Transformer ......................... clip/model.py:404-440
  VisionTransformer_MuDPT ............. clip/model.py:499-553
  CLIP ................................ clip/model.py:667-854
  build_model ......................... clip/model.py:881-921
"""
from __future__ import annotations

import math
from collections import OrderedDict
from typing import Dict, Optional

import numpy as np
import torch
import torch.nn.functional as F
from torch import nn

from ..engine import Engine, vision_tower


def _cfg_get(cfg, key: str):
    """cfg.TRAINER.<NAME>.<key> (the reference evaluates this string, clip/model.py:268)."""
    name = str(cfg.TRAINER.NAME).upper()
    node = cfg.TRAINER[name] if isinstance(cfg.TRAINER, dict) else getattr(cfg.TRAINER, name)
    return node[key] if isinstance(node, dict) else getattr(node, key)


class LayerNorm(nn.LayerNorm):
    """Container for gamma/beta; the native LayerNorm kernels compute in fp32 (clip/model.py:164-170)."""


class QuickGELU(nn.Module):
    """Placeholder in `mlp` so that state-dict keys match; QuickGELU is fused into the c_fc GEMM epilogue."""

    def forward(self, x):  # pragma: no cover - never on the hot path
        raise NotImplementedError("QuickGELU runs fused inside the native c_fc GEMM epilogue")


class ResidualAttentionBlock_MuDPT(nn.Module):
    def __init__(self, d_model: int, n_head: int, attn_mask: torch.Tensor = None, nth_layer: int = 0,
                 is_text_layer: bool = False, cfg=None):
        super().__init__()
        self.attn = nn.MultiheadAttention(d_model, n_head)
        self.ln_1 = LayerNorm(d_model)
        self.mlp = nn.Sequential(OrderedDict([
            ("c_fc", nn.Linear(d_model, d_model * 4)),
            ("gelu", QuickGELU()),
            ("c_proj", nn.Linear(d_model * 4, d_model)),
        ]))
        self.ln_2 = LayerNorm(d_model)
        self.attn_mask = attn_mask
        self.is_text_layer = is_text_layer
        self.prompt_nctx = _cfg_get(cfg, "N_CTX")
        self.is_first_layer = nth_layer == 0

    def forward(self, inputs):  # pragma: no cover
        raise NotImplementedError("blocks run fused inside the native tower (mudpt_vision_forward / mudpt_text_forward)")


class ResidualAttentionBlock(nn.Module):
    """Plain block (clip/model.py:178-199): the cfg=None CLIP that CoCoOp builds on (trainers/cocoop.py:34)."""

    def __init__(self, d_model: int, n_head: int, attn_mask: torch.Tensor = None):
        super().__init__()
        self.attn = nn.MultiheadAttention(d_model, n_head)
        self.ln_1 = LayerNorm(d_model)
        self.mlp = nn.Sequential(OrderedDict([
            ("c_fc", nn.Linear(d_model, d_model * 4)),
            ("gelu", QuickGELU()),
            ("c_proj", nn.Linear(d_model * 4, d_model)),
        ]))
        self.ln_2 = LayerNorm(d_model)
        self.attn_mask = attn_mask

    def forward(self, x):  # pragma: no cover
        raise NotImplementedError("blocks run fused inside the native tower (mudpt_vision_forward / mudpt_text_forward)")


class Transformer(nn.Module):
    def __init__(self, width: int, layers: int, heads: int, attn_mask: torch.Tensor = None, prompt_depth: int = 0,
                 is_text_layer: bool = False, cfg=None):
        super().__init__()
        self.width, self.layers, self.heads = width, layers, heads
        if cfg is None:  # clip/model.py:436-437
            self.resblocks = nn.Sequential(*[ResidualAttentionBlock(width, heads, attn_mask) for _ in range(layers)])
            return
        if cfg.TRAINER.NAME not in ("MuDPT", "UMuDPT", "UUMuDPT"):
            raise NotImplementedError(f"{getattr(getattr(cfg, 'TRAINER', None), 'NAME', None)} is not implemented")
        # the UMuDPT / UUMuDPT blocks (clip/model.py:302-400) splice exactly like the MuDPT block (:275-301)
        self.resblocks = nn.Sequential(*[
            ResidualAttentionBlock_MuDPT(width, heads, attn_mask, i, is_text_layer, cfg=cfg) for i in range(layers)])

    def forward(self, x):  # pragma: no cover
        raise NotImplementedError("the tower runs natively; call the owning encoder")


class VisionTransformer_MuDPT(nn.Module):
    def __init__(self, input_resolution: int, patch_size: int, width: int, layers: int, heads: int, output_dim: int, cfg=None):
        super().__init__()
        self.input_resolution = input_resolution
        self.output_dim = output_dim
        self.conv1 = nn.Conv2d(in_channels=3, out_channels=width, kernel_size=patch_size, stride=patch_size, bias=False)
        scale = width ** -0.5
        self.class_embedding = nn.Parameter(scale * torch.randn(width))
        self.positional_embedding = nn.Parameter(scale * torch.randn((input_resolution // patch_size) ** 2 + 1, width))
        self.deep_prompts_depth = _cfg_get(cfg, "DEEP_PROMPT_DEPTH")
        n_ctx = _cfg_get(cfg, "N_CTX")
        self.visual_ctx = nn.Parameter(torch.empty(n_ctx, width).normal_(std=0.02))
        self.visual_ctx_deep_prompts = nn.Parameter(torch.empty(self.deep_prompts_depth - 1, n_ctx, width).normal_(std=0.02))
        self.visual_ctx_deep_projections = nn.Linear(in_features=width, out_features=output_dim)
        self.ln_pre = LayerNorm(width)
        self.transformer = Transformer(width, layers, heads, cfg=cfg)
        self.ln_post = LayerNorm(width)
        self.proj = nn.Parameter(scale * torch.randn(width, output_dim))
        self._owner = None  # set by CLIP: gives access to the shared native engine

    def prompt_stack(self, shared_prompt, t2v_visual_prompts):
        """[depth, n_ctx, width]: row block 0 is the layer-0 prompt after ln_pre (clip/model.py:534-541),
        blocks 1.. are t2v + visual deep prompts (:537).  Tiny differentiable torch ops."""
        shallow = self.visual_ctx.unsqueeze(0) + shared_prompt            # [1, n, width]
        p0 = F.layer_norm(shallow.float(), (shallow.shape[-1],), self.ln_pre.weight.float(), self.ln_pre.bias.float(),
                          self.ln_pre.eps)
        deep = t2v_visual_prompts + self.visual_ctx_deep_prompts           # [depth-1, n, width]
        return torch.cat([p0, deep.float()], dim=0)

    def forward(self, x: torch.Tensor, shared_prompt, t2v_visual_prompts):
        engine = self._owner().engine(x.device)
        text_prompts = self.visual_ctx_deep_projections(self.visual_ctx_deep_prompts)   # v2t, clip/model.py:539
        feats = vision_tower(engine, x, self.prompt_stack(shared_prompt, t2v_visual_prompts))
        return feats, text_prompts


class LightTransformer(nn.Module):
    """One plain block over the handful of prompt tokens (trainers/umudpt.py:56-79, clip/model.py:203-226): the only
    part of the UMuDPT / UUMuDPT variants that is not a frozen tower.  [n_ctx x depth] tokens -- real torch modules
    under autograd (this is trainable prompt algebra, like the three Linear layers of MuDPT)."""

    def __init__(self, d_model: int, n_head: int, attn_mask: torch.Tensor = None):
        super().__init__()
        self.attn = nn.MultiheadAttention(d_model, n_head)
        self.ln_1 = nn.LayerNorm(d_model)
        self.mlp = nn.Sequential(OrderedDict([
            ("c_fc", nn.Linear(d_model, d_model * 4)),
            ("gelu", _QuickGELUTorch()),
            ("c_proj", nn.Linear(d_model * 4, d_model)),
        ]))
        self.ln_2 = nn.LayerNorm(d_model)
        self.attn_mask = attn_mask

    def forward(self, x: torch.Tensor):
        a = self.ln_1(x)
        x = x + self.attn(a, a, a, need_weights=False, attn_mask=self.attn_mask)[0]
        return x + self.mlp(self.ln_2(x))


class _QuickGELUTorch(nn.Module):
    def forward(self, x):
        return x * torch.sigmoid(1.702 * x)


def _stack_with_ln_pre(vit, shared_ctx, deeper_prompts):
    """[depth, n_ctx, width]: row block 0 = ln_pre(shared ctx) (the ctx rows are appended before ln_pre,
    clip/model.py:578-581), blocks 1.. = the deep visual prompts."""
    p0 = F.layer_norm(shared_ctx.float(), (shared_ctx.shape[-1],), vit.ln_pre.weight.float(), vit.ln_pre.bias.float(),
                      vit.ln_pre.eps)
    return torch.cat([p0, deeper_prompts.float()], dim=0)


class VisionTransformer_UMuDPT(nn.Module):
    """clip/model.py:556-597: no trainable tensor of its own; forward(x, shared_ctx [1,n,w], deeper [D-1,n,w])."""

    def __init__(self, input_resolution: int, patch_size: int, width: int, layers: int, heads: int, output_dim: int, cfg=None):
        super().__init__()
        self.input_resolution = input_resolution
        self.output_dim = output_dim
        self.conv1 = nn.Conv2d(in_channels=3, out_channels=width, kernel_size=patch_size, stride=patch_size, bias=False)
        scale = width ** -0.5
        self.class_embedding = nn.Parameter(scale * torch.randn(width))
        self.positional_embedding = nn.Parameter(scale * torch.randn((input_resolution // patch_size) ** 2 + 1, width))
        self.deep_prompts_depth = _cfg_get(cfg, "DEEP_PROMPT_DEPTH")
        self.ln_pre = LayerNorm(width)
        self.transformer = Transformer(width, layers, heads, cfg=cfg)
        self.ln_post = LayerNorm(width)
        self.proj = nn.Parameter(scale * torch.randn(width, output_dim))
        self._owner = None

    def forward(self, x: torch.Tensor, shared_ctx, deeper_prompts):
        engine = self._owner().engine(x.device)
        return vision_tower(engine, x, _stack_with_ln_pre(self, shared_ctx, deeper_prompts))


class VisionTransformer_UUMuDPT(nn.Module):
    """clip/model.py:600-664: UMuDPT plus vision-side prompts and their LightTransformer -> text prompts."""

    def __init__(self, input_resolution: int, patch_size: int, width: int, layers: int, heads: int, output_dim: int, cfg=None):
        super().__init__()
        self.input_resolution = input_resolution
        self.output_dim = output_dim
        self.conv1 = nn.Conv2d(in_channels=3, out_channels=width, kernel_size=patch_size, stride=patch_size, bias=False)
        scale = width ** -0.5
        self.class_embedding = nn.Parameter(scale * torch.randn(width))
        self.positional_embedding = nn.Parameter(scale * torch.randn((input_resolution // patch_size) ** 2 + 1, width))
        self.deep_prompts_depth = _cfg_get(cfg, "DEEP_PROMPT_DEPTH")
        n_ctx = _cfg_get(cfg, "N_CTX")
        self.visual_ctx = nn.Parameter(torch.empty(n_ctx, width).normal_(std=0.02))
        self.visual_ctx_deep_prompts = nn.Parameter(torch.empty(self.deep_prompts_depth - 1, n_ctx, width).normal_(std=0.02))
        self.visual_ctx_ln_intra_pre = nn.LayerNorm(width)
        self.visual_ctx_self_attn = LightTransformer(d_model=width, n_head=width // 64)
        self.visual_ctx_ln_intra_post = nn.LayerNorm(width)
        self.visual_ctx_text_proj = nn.Linear(in_features=width, out_features=output_dim)
        self.ln_pre = LayerNorm(width)
        self.transformer = Transformer(width, layers, heads, cfg=cfg)
        self.ln_post = LayerNorm(width)
        self.proj = nn.Parameter(scale * torch.randn(width, output_dim))
        self._owner = None

    def textual_prompts(self):
        t = self.visual_ctx_ln_intra_pre(self.visual_ctx_deep_prompts)
        t = self.visual_ctx_self_attn(t.permute(1, 0, 2)).permute(1, 0, 2)
        return self.visual_ctx_text_proj(self.visual_ctx_ln_intra_post(t))

    def forward(self, x: torch.Tensor, shared_ctx, deeper_prompts):
        engine = self._owner().engine(x.device)
        shared = shared_ctx + self.visual_ctx.unsqueeze(0)
        deeper = deeper_prompts + self.visual_ctx_deep_prompts
        feats = vision_tower(engine, x, _stack_with_ln_pre(self, shared, deeper))
        return feats, self.textual_prompts()


class VisionTransformer(nn.Module):
    """Plain ViT tower without image prompts (clip/model.py:443-496, cfg=None): same parameter names;
    forward(x) -> image features through the native tower (no trainable tensor inside: differentiable w.r.t. x only)."""

    def __init__(self, input_resolution: int, patch_size: int, width: int, layers: int, heads: int, output_dim: int, cfg=None):
        super().__init__()
        self.input_resolution = input_resolution
        self.output_dim = output_dim
        self.conv1 = nn.Conv2d(in_channels=3, out_channels=width, kernel_size=patch_size, stride=patch_size, bias=False)
        scale = width ** -0.5
        self.class_embedding = nn.Parameter(scale * torch.randn(width))
        self.positional_embedding = nn.Parameter(scale * torch.randn((input_resolution // patch_size) ** 2 + 1, width))
        self.img_prompt_depth, self.img_prompt = 0, False
        self.ln_pre = LayerNorm(width)
        self.transformer = Transformer(width, layers, heads, cfg=None)
        self.ln_post = LayerNorm(width)
        self.proj = nn.Parameter(scale * torch.randn(width, output_dim))
        self._owner = None

    def forward(self, x: torch.Tensor):
        engine = self._owner().engine(x.device)
        empty = torch.zeros(engine.depth, 0, self.conv1.weight.shape[0], device=x.device, dtype=torch.float32)
        # the tower is frozen and carries no prompts: the forward-only walk unless x itself requires a gradient
        return vision_tower(engine, x, empty)


class CLIP(nn.Module):
    def __init__(self, embed_dim: int, image_resolution: int, vision_layers: int, vision_width: int,
                 vision_patch_size: int, context_length: int, vocab_size: int, transformer_width: int,
                 transformer_heads: int, transformer_layers: int, cfg=None):
        super().__init__()
        if isinstance(vision_layers, (tuple, list)):
            raise NotImplementedError("ModifiedResNet towers are outside the MuDPT ViT hot path")
        if cfg is not None and cfg.TRAINER.NAME not in ("MuDPT", "UMuDPT", "UUMuDPT"):
            raise NotImplementedError("implemented: cfg.TRAINER.NAME in MuDPT / UMuDPT / UUMuDPT and the plain cfg=None model")
        self.context_length = context_length
        self.arch = dict(embed_dim=embed_dim, image_resolution=image_resolution, vision_layers=vision_layers,
                         vision_width=vision_width, vision_patch_size=vision_patch_size, context_length=context_length,
                         vocab_size=vocab_size, transformer_width=transformer_width, transformer_heads=transformer_heads,
                         transformer_layers=transformer_layers)
        # cfg=None: plain towers (clip/model.py:742-750) -> a native handle without spliced prompts
        self.n_ctx = _cfg_get(cfg, "N_CTX") if cfg is not None else 0
        self.depth = _cfg_get(cfg, "DEEP_PROMPT_DEPTH") if cfg is not None else 1
        vit = VisionTransformer if cfg is None else {"MuDPT": VisionTransformer_MuDPT, "UMuDPT": VisionTransformer_UMuDPT,
                                                     "UUMuDPT": VisionTransformer_UUMuDPT}[cfg.TRAINER.NAME]
        self.visual = vit(input_resolution=image_resolution, patch_size=vision_patch_size, width=vision_width,
                          layers=vision_layers, heads=vision_width // 64, output_dim=embed_dim, cfg=cfg)
        self.transformer = Transformer(width=transformer_width, layers=transformer_layers, heads=transformer_heads,
                                       attn_mask=None, is_text_layer=True, cfg=cfg)
        self.vocab_size = vocab_size
        self.token_embedding = nn.Embedding(vocab_size, transformer_width)
        self.positional_embedding = nn.Parameter(torch.empty(self.context_length, transformer_width))
        self.ln_final = LayerNorm(transformer_width)
        self.text_projection = nn.Parameter(torch.empty(transformer_width, embed_dim))
        self.logit_scale = nn.Parameter(torch.ones([]) * np.log(1 / 0.07))
        self.initialize_parameters()
        import weakref
        self.visual._owner = weakref.ref(self)
        self._engine: Optional[Engine] = None

    def initialize_parameters(self):
        """Same distributions as clip/model.py:781-808 (text tower only; the vision tower keeps torch defaults)."""
        nn.init.normal_(self.token_embedding.weight, std=0.02)
        nn.init.normal_(self.positional_embedding, std=0.01)
        proj_std = (self.transformer.width ** -0.5) * ((2 * self.transformer.layers) ** -0.5)
        attn_std = self.transformer.width ** -0.5
        fc_std = (2 * self.transformer.width) ** -0.5
        for block in self.transformer.resblocks:
            nn.init.normal_(block.attn.in_proj_weight, std=attn_std)
            nn.init.normal_(block.attn.out_proj.weight, std=proj_std)
            nn.init.normal_(block.mlp.c_fc.weight, std=fc_std)
            nn.init.normal_(block.mlp.c_proj.weight, std=proj_std)
        nn.init.normal_(self.text_projection, std=self.transformer.width ** -0.5)

    @property
    def dtype(self):
        return self.visual.conv1.weight.dtype

    # ---- native engine (lazy: needs the module to live on a CUDA device) ----
    def engine(self, device=None) -> Engine:
        device = torch.device(device) if device is not None else self.visual.conv1.weight.device
        if self._engine is None or self._engine.device != device:
            if device.type != "cuda":
                raise RuntimeError("mudpt_b200: the MuDPT hot path needs a CUDA (sm_100a) device; there is no CPU fallback")
            eng = Engine(self.arch, self.n_ctx, self.depth, device)
            eng.load_clip_weights({k: v for k, v in self.state_dict().items()})
            self._engine = eng
        return self._engine

    def refresh_engine_weights(self):
        """Call after load_state_dict() if the frozen CLIP weights changed."""
        if self._engine is not None:
            self._engine.load_clip_weights({k: v for k, v in self.state_dict().items()})


def build_model(state_dict: Dict[str, torch.Tensor], cfg=None) -> CLIP:
    """Shape inference from a CLIP state dict, ViT towers only (clip/model.py:881-921)."""
    if "visual.proj" not in state_dict:
        raise NotImplementedError("ResNet CLIP checkpoints are outside the MuDPT ViT hot path")
    vision_width = state_dict["visual.conv1.weight"].shape[0]
    vision_layers = len([k for k in state_dict if k.startswith("visual.") and k.endswith(".attn.in_proj_weight")])
    vision_patch_size = state_dict["visual.conv1.weight"].shape[-1]
    grid_size = round((state_dict["visual.positional_embedding"].shape[0] - 1) ** 0.5)
    image_resolution = vision_patch_size * grid_size
    embed_dim = state_dict["text_projection"].shape[1]
    context_length = state_dict["positional_embedding"].shape[0]
    vocab_size = state_dict["token_embedding.weight"].shape[0]
    transformer_width = state_dict["ln_final.weight"].shape[0]
    transformer_heads = transformer_width // 64
    transformer_layers = len(set(k.split(".")[2] for k in state_dict if k.startswith("transformer.resblocks")))
    model = CLIP(embed_dim, image_resolution, vision_layers, vision_width, vision_patch_size, context_length,
                 vocab_size, transformer_width, transformer_heads, transformer_layers, cfg)
    sd = {k: v for k, v in state_dict.items() if k not in ("input_resolution", "context_length", "vocab_size")}
    model.load_state_dict(sd, strict=False)
    return model.eval()

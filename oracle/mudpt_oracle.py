"""TEST INFRASTRUCTURE ONLY -- fp32 CPU restatement of the MuDPT hot path.

This is the oracle the CUDA path is checked against.  It restates, in plain fp32 torch
ops on explicit weight tensors (no nn.MultiheadAttention / nn.LayerNorm modules), the
math of the reference:

  * LayerNorm / QuickGELU ............ clip/model.py:164-175
  * residual block + prompt splice .... clip/model.py:254-301 (MHA call :271-273)
  * causal mask ....................... clip/model.py:810-816
  * vision tower ...................... clip/model.py:526-553
  * prompt learner .................... trainers/mudpt.py:97-130
  * text tower + EOT gather ........... trainers/mudpt.py:142-156
  * cosine logits ..................... trainers/mudpt.py:170-184
  * loss .............................. trainers/mudpt.py:250 (F.cross_entropy, mean)

The arithmetic of the reference lives in third-party PyTorch (unpinned by the reference;
torch 2.11.0 CPU here).  Parity pinning: `tests/test_oracle.py` runs the
*reference itself* (imported read-only under oracle/ref_shims.py) against this file when
MUDPT_REFERENCE_ROOT names a checkout of it, and `tests/golden/*.npz` (made by oracle/make_golden.py from the
reference) pins it everywhere else.  The reference has no tests / golden vectors of its own
(SURVEY.md section 4).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module.  Nothing under mudpt_b200/ does.

Weights are a flat dict keyed by the reference CustomCLIP.state_dict() names.
Layout here is NLD ([sequence, token, width]); the reference uses LND -- a pure permutation.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import torch
import torch.nn.functional as F

TRAINABLE = (
    "mudpt_prompt_learner.ctx",
    "mudpt_prompt_learner.deep_prompts",
    "mudpt_prompt_learner.embed_projection.weight",
    "mudpt_prompt_learner.embed_projection.bias",
    "mudpt_prompt_learner.deep_projections.weight",
    "mudpt_prompt_learner.deep_projections.bias",
    "image_encoder.visual_ctx",
    "image_encoder.visual_ctx_deep_prompts",
    "image_encoder.visual_ctx_deep_projections.weight",
    "image_encoder.visual_ctx_deep_projections.bias",
)


def layer_norm(x, w, b, eps: float = 1e-5):
    """clip/model.py:164-170 -- fp32 LN, biased variance."""
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    return (x - mu) * torch.rsqrt(var + eps) * w + b


def quick_gelu(x):
    """clip/model.py:173-175."""
    return x * torch.sigmoid(1.702 * x)


def causal_mask(L: int, dtype=torch.float32):
    """clip/model.py:810-816 -- additive mask, -inf strictly above the diagonal."""
    return torch.full((L, L), float("-inf"), dtype=dtype).triu_(1)


def attention(x, w_in, b_in, w_out, b_out, n_head: int, mask: Optional[torch.Tensor]):
    """nn.MultiheadAttention as called at clip/model.py:271-273 (packed in-proj, heads of
    width d/n_head, scale 1/sqrt(dh), additive mask, softmax over keys, out-proj)."""
    N, L, d = x.shape
    dh = d // n_head
    qkv = x @ w_in.t() + b_in
    q, k, v = qkv.split(d, dim=-1)
    q = q.view(N, L, n_head, dh).transpose(1, 2)
    k = k.view(N, L, n_head, dh).transpose(1, 2)
    v = v.view(N, L, n_head, dh).transpose(1, 2)
    s = (q @ k.transpose(-1, -2)) * (1.0 / math.sqrt(dh))
    if mask is not None:
        s = s + mask
    p = torch.softmax(s, dim=-1)
    o = (p @ v).transpose(1, 2).reshape(N, L, d)
    return o @ w_out.t() + b_out


def block(x, sd: Dict[str, torch.Tensor], pfx: str, n_head: int, mask):
    """clip/model.py:299-300."""
    a = layer_norm(x, sd[pfx + "ln_1.weight"], sd[pfx + "ln_1.bias"])
    x = x + attention(a, sd[pfx + "attn.in_proj_weight"], sd[pfx + "attn.in_proj_bias"],
                      sd[pfx + "attn.out_proj.weight"], sd[pfx + "attn.out_proj.bias"], n_head, mask)
    m = layer_norm(x, sd[pfx + "ln_2.weight"], sd[pfx + "ln_2.bias"])
    h = m @ sd[pfx + "mlp.c_fc.weight"].t() + sd[pfx + "mlp.c_fc.bias"]
    x = x + quick_gelu(h) @ sd[pfx + "mlp.c_proj.weight"].t() + sd[pfx + "mlp.c_proj.bias"]
    return x


def tower(x, deep, sd, pfx: str, n_layers: int, n_head: int, mask, row0: int, n_ctx: int):
    """Transformer of ResidualAttentionBlock_MuDPT (clip/model.py:275-301, 418-421):
    layer i in 1..deep.shape[0] overwrites rows [row0, row0+n_ctx) with deep[i-1] first."""
    for i in range(n_layers):
        if i > 0 and (i - 1) < deep.shape[0]:
            x = torch.cat([x[:, :row0], deep[i - 1].unsqueeze(0).expand(x.shape[0], -1, -1),
                           x[:, row0 + n_ctx:]], dim=1)
        x = block(x, sd, f"{pfx}resblocks.{i}.", n_head, mask)
    return x


def count_layers(sd, pfx: str) -> int:
    n = 0
    while f"{pfx}resblocks.{n}.ln_1.weight" in sd:
        n += 1
    return n


def prompt_learner(sd):
    """trainers/mudpt.py:117-130 (+ construct_prompts :97-115)."""
    P = "mudpt_prompt_learner."
    ctx = sd[P + "ctx"]
    prefix, suffix = sd[P + "token_prefix"], sd[P + "token_suffix"]
    C = prefix.shape[0]
    prompts = torch.cat([prefix, ctx.unsqueeze(0).expand(C, -1, -1), suffix], dim=1)
    deep = sd[P + "deep_prompts"]
    visual_prompts = deep @ sd[P + "deep_projections.weight"].t() + sd[P + "deep_projections.bias"]
    shared = ctx.unsqueeze(0) @ sd[P + "embed_projection.weight"].t() + sd[P + "embed_projection.bias"]
    return prompts, shared, deep, visual_prompts


def vision_tower(sd, image, shared_prompt, t2v_visual_prompts, n_head: Optional[int] = None):
    """VisionTransformer_MuDPT.forward, clip/model.py:526-553."""
    V = "image_encoder."
    w = sd[V + "conv1.weight"]
    width, patch = w.shape[0], w.shape[-1]
    n_head = n_head or width // 64
    x = F.conv2d(image, w, stride=patch)
    x = x.reshape(x.shape[0], width, -1).permute(0, 2, 1)
    cls = sd[V + "class_embedding"].expand(x.shape[0], 1, width)
    x = torch.cat([cls, x], dim=1) + sd[V + "positional_embedding"]
    vctx = sd[V + "visual_ctx"]
    n_ctx = vctx.shape[0]
    vp = (vctx.unsqueeze(0) + shared_prompt).expand(x.shape[0], -1, -1)
    x = torch.cat([x, vp], dim=1)
    vdeep = sd[V + "visual_ctx_deep_prompts"]
    visual_deep = t2v_visual_prompts + vdeep
    text_prompts = vdeep @ sd[V + "visual_ctx_deep_projections.weight"].t() + sd[V + "visual_ctx_deep_projections.bias"]
    x = layer_norm(x, sd[V + "ln_pre.weight"], sd[V + "ln_pre.bias"])
    L = x.shape[1]
    x = tower(x, visual_deep, sd, V + "transformer.", count_layers(sd, V + "transformer."), n_head,
              None, L - n_ctx, n_ctx)
    x = layer_norm(x[:, 0, :], sd[V + "ln_post.weight"], sd[V + "ln_post.bias"])
    return x @ sd[V + "proj"], text_prompts


def text_tower(sd, prompts, eot, deep_prompts, n_head: Optional[int] = None, n_ctx: Optional[int] = None):
    """TextEncoder.forward, trainers/mudpt.py:142-156.  `eot` = argmax of the token ids."""
    T = "text_encoder."
    d = prompts.shape[-1]
    n_head = n_head or d // 64
    n_ctx = n_ctx if n_ctx is not None else sd["mudpt_prompt_learner.ctx"].shape[0]
    L = prompts.shape[1]
    x = prompts + sd[T + "positional_embedding"][:L]
    x = tower(x, deep_prompts, sd, T + "transformer.", count_layers(sd, T + "transformer."), n_head,
              causal_mask(L), 1, n_ctx)
    x = layer_norm(x, sd[T + "ln_final.weight"], sd[T + "ln_final.bias"])
    x = x[torch.arange(x.shape[0]), eot]
    return x @ sd[T + "text_projection"]


def forward(sd, image, tokenized_prompts, labels=None):
    """CustomCLIP.forward (trainers/mudpt.py:170-184) (+ CE of :250 when labels given)."""
    prompts, shared, text_deep, t2v = prompt_learner(sd)
    f_img, v2t = vision_tower(sd, image, shared, t2v)
    text_prompts = text_deep + v2t
    eot = tokenized_prompts.argmax(dim=-1).long()
    f_txt = text_tower(sd, prompts, eot, text_prompts)
    fi = f_img / f_img.norm(dim=-1, keepdim=True)
    ft = f_txt / f_txt.norm(dim=-1, keepdim=True)
    logits = sd["logit_scale"].exp() * fi @ ft.t()
    out = {"logits": logits, "image_features": f_img, "text_features": f_txt}
    if labels is not None:
        out["loss"] = F.cross_entropy(logits, labels)
    return out


def forward_backward(sd, image, tokenized_prompts, labels):
    """One train step's tensors: forward + autograd of the 10 trainable tensors
    (freeze rule trainers/mudpt.py:205-212).  Returns detached results + grads."""
    sd = dict(sd)
    leaves = {}
    for k in TRAINABLE:
        leaves[k] = sd[k].detach().clone().requires_grad_(True)
        sd[k] = leaves[k]
    out = forward(sd, image, tokenized_prompts, labels)
    grads = torch.autograd.grad(out["loss"], [leaves[k] for k in TRAINABLE], allow_unused=True)
    res = {k: v.detach() for k, v in out.items()}
    # depth == 1: the deep tensors (leading dim 0) and their projections are unused -> zero grad
    res["grads"] = {k: (g.detach() if g is not None else torch.zeros_like(leaves[k]))
                    for k, g in zip(TRAINABLE, grads)}
    return res


# ---------------------------------------------------------------------------------------------
# Synthetic inputs (SURVEY.md section 8d).  Pure functions of a seed; used by the golden
# generator, the parity tests and the bench's CPU leg.
# ---------------------------------------------------------------------------------------------

def synthetic_images(batch: int, size: int = 224, seed: int = 1, kind: str = "noise"):
    g = torch.Generator().manual_seed(seed)
    if kind == "noise":
        return torch.randn(batch, 3, size, size, generator=g)
    if kind == "colour":  # constant-colour images: per-image structure (SURVEY.md H1)
        return torch.randn(batch, 3, 1, 1, generator=g).expand(batch, 3, size, size).contiguous()
    raise ValueError(kind)


def synthetic_labels(batch: int, n_cls: int, seed: int = 1):
    g = torch.Generator().manual_seed(seed + 1000)
    return torch.randint(0, n_cls, (batch,), generator=g)


def metrics(a: torch.Tensor, b: torch.Tensor):
    """cosine, rel-L2 and max-abs error of a against b (flattened)."""
    a = a.double().flatten()
    b = b.double().flatten()
    cos = float((a @ b) / (a.norm() * b.norm() + 1e-300))
    rel = float((a - b).norm() / (b.norm() + 1e-300))
    return {"cos": cos, "rel_l2": rel, "max_abs": float((a - b).abs().max())}


def top1_agreement(logits: torch.Tensor, ref_logits: torch.Tensor, err: float):
    """Raw and margin-aware top-1 agreement (SURVEY.md H1): a row is 'decidable' when the
    fp32 top-1/top-2 margin exceeds 2*err."""
    top2 = ref_logits.topk(2, dim=-1).values
    margin = top2[:, 0] - top2[:, 1]
    agree = logits.argmax(-1) == ref_logits.argmax(-1)
    dec = margin > 2 * err
    return {"raw": float(agree.float().mean()),
            "decidable_frac": float(dec.float().mean()),
            "margin_aware": float(agree[dec].float().mean()) if dec.any() else 1.0}


# ---------------------------------------------------------------------------------------------
# "Prompt stack" form of the towers: the exact decomposition the C ABI uses
# (include/mudpt_b200.h): stack[0] = layer-0 prompt rows, stack[i>=1] = deep prompts of layer i.
# Used by tests to emulate the native engine on CPU (tests/fake_engine.py).
# ---------------------------------------------------------------------------------------------

def tower_stack(x, stack, sd, pfx, n_layers, n_head, mask, row0, first_splice=0):
    n_ctx = stack.shape[1]
    for i in range(n_layers):
        if first_splice <= i < stack.shape[0] and n_ctx > 0:
            x = torch.cat([x[:, :row0], stack[i].unsqueeze(0).expand(x.shape[0], -1, -1), x[:, row0 + n_ctx:]], dim=1)
        x = block(x, sd, f"{pfx}resblocks.{i}.", n_head, mask)
    return x


def vision_features_from_stack(sd, image, stack):
    """mudpt_vision_forward: images + [depth, n, dv] stack (stack[0] already ln_pre'd) -> f_img."""
    V = "image_encoder."
    w = sd[V + "conv1.weight"]
    width, patch = w.shape[0], w.shape[-1]
    x = F.conv2d(image, w, stride=patch)
    x = x.reshape(x.shape[0], width, -1).permute(0, 2, 1)
    x = torch.cat([sd[V + "class_embedding"].expand(x.shape[0], 1, width), x], dim=1) + sd[V + "positional_embedding"]
    x = layer_norm(x, sd[V + "ln_pre.weight"], sd[V + "ln_pre.bias"])
    n = stack.shape[1]
    x = torch.cat([x, torch.zeros(x.shape[0], n, width)], dim=1)
    x = tower_stack(x, stack, sd, V + "transformer.", count_layers(sd, V + "transformer."), width // 64, None,
                    x.shape[1] - n)
    return layer_norm(x[:, 0, :], sd[V + "ln_post.weight"], sd[V + "ln_post.bias"]) @ sd[V + "proj"]


def text_features_from_stack(sd, embeddings, eot, stack, seq_len, first_splice=0):
    """mudpt_text_forward: token embeddings [C, >=seq_len, dt] (ctx rows ignored when
    first_splice == 0) + [depth, n, dt] stack -> f_txt."""
    T = "text_encoder."
    d = embeddings.shape[-1]
    x = embeddings[:, :seq_len] + sd[T + "positional_embedding"][:seq_len]
    x = tower_stack(x, stack, sd, T + "transformer.", count_layers(sd, T + "transformer."), d // 64,
                    causal_mask(seq_len), 1, first_splice)
    x = layer_norm(x, sd[T + "ln_final.weight"], sd[T + "ln_final.bias"])
    return x[torch.arange(x.shape[0]), eot] @ sd[T + "text_projection"]


def logits_and_loss(f_img, f_txt, logit_scale, labels=None, inv_global_batch=None):
    fi = f_img / f_img.norm(dim=-1, keepdim=True)
    ft = f_txt / f_txt.norm(dim=-1, keepdim=True)
    logits = logit_scale.exp() * fi @ ft.t()
    if labels is None:
        return logits, None
    loss = F.cross_entropy(logits, labels, reduction="sum") * inv_global_batch
    return logits, loss

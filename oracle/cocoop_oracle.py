"""TEST INFRASTRUCTURE ONLY -- fp32 CPU restatement of the reference CoCoOp path
(BASELINE config 4: instance-conditioned prompts on the plain CLIP towers).

Only tests/, __graft_entry__.smoke() and bench.py's CPU leg may import this file; the product
(mudpt_b200/) never does.  Pinned against the reference itself: tests/golden/cocoop_*.npz are
produced by oracle/make_golden.py from the unmodified trainers/cocoop.py, and
tests/test_oracle.py checks this restatement against them (and against the live reference when
MUDPT_REFERENCE_ROOT names a checkout of it).

  PromptLearner.forward ... trainers/cocoop.py:149-163     (ctx + meta_net(im_features), per image)
  TextEncoder.forward ..... trainers/cocoop.py:52-64       (plain blocks, clip/model.py:178-199)
  VisionTransformer ....... clip/model.py:474-496          (plain)
  CustomCLIP.forward ...... trainers/cocoop.py:176-198
"""
from __future__ import annotations

from typing import Dict

import torch
import torch.nn.functional as F

from .mudpt_oracle import causal_mask, count_layers, layer_norm, tower

TRAINABLE = ("prompt_learner.ctx", "prompt_learner.meta_net.linear1.weight", "prompt_learner.meta_net.linear1.bias",
             "prompt_learner.meta_net.linear2.weight", "prompt_learner.meta_net.linear2.bias")


def _no_deep(d):
    return torch.zeros(0, 0, d)


def vision_tower(sd, image):
    """VisionTransformer.forward without image prompts (clip/model.py:474-496)."""
    V = "image_encoder."
    w = sd[V + "conv1.weight"]
    width, patch = w.shape[0], w.shape[-1]
    x = F.conv2d(image, w, stride=patch)
    x = x.reshape(x.shape[0], width, -1).permute(0, 2, 1)
    x = torch.cat([sd[V + "class_embedding"].expand(x.shape[0], 1, width), x], dim=1) + sd[V + "positional_embedding"]
    x = layer_norm(x, sd[V + "ln_pre.weight"], sd[V + "ln_pre.bias"])
    x = tower(x, _no_deep(width), sd, V + "transformer.", count_layers(sd, V + "transformer."), width // 64, None, 0, 0)
    x = layer_norm(x[:, 0, :], sd[V + "ln_post.weight"], sd[V + "ln_post.bias"])
    return x @ sd[V + "proj"]


def text_tower(sd, prompts, eot):
    """TextEncoder.forward (trainers/cocoop.py:52-64)."""
    T = "text_encoder."
    d, L = prompts.shape[-1], prompts.shape[1]
    x = prompts + sd[T + "positional_embedding"][:L]
    x = tower(x, _no_deep(d), sd, T + "transformer.", count_layers(sd, T + "transformer."), d // 64, causal_mask(L), 0, 0)
    x = layer_norm(x, sd[T + "ln_final.weight"], sd[T + "ln_final.bias"])
    return x[torch.arange(x.shape[0]), eot] @ sd[T + "text_projection"]


def prompt_learner(sd, im_features):
    """[B, C, 77, d] instance-conditioned prompts (trainers/cocoop.py:149-163)."""
    P = "prompt_learner."
    h = torch.relu(im_features @ sd[P + "meta_net.linear1.weight"].t() + sd[P + "meta_net.linear1.bias"])
    bias = h @ sd[P + "meta_net.linear2.weight"].t() + sd[P + "meta_net.linear2.bias"]      # [B, d]
    ctx = sd[P + "ctx"].unsqueeze(0) + bias.unsqueeze(1)                                     # [B, n_ctx, d]
    prefix, suffix = sd[P + "token_prefix"], sd[P + "token_suffix"]
    C = prefix.shape[0]
    return torch.stack([torch.cat([prefix, c.unsqueeze(0).expand(C, -1, -1), suffix], dim=1) for c in ctx])


def forward(sd, image, tokenized_prompts, labels=None):
    f_img = vision_tower(sd, image)
    fi = f_img / f_img.norm(dim=-1, keepdim=True)
    prompts = prompt_learner(sd, fi)
    eot = tokenized_prompts.argmax(dim=-1).long()
    scale = sd["logit_scale"].exp()
    logits, feats = [], []
    for pts_i, imf_i in zip(prompts, fi):
        tf = text_tower(sd, pts_i, eot)
        feats.append(tf)
        tf = tf / tf.norm(dim=-1, keepdim=True)
        logits.append(scale * imf_i @ tf.t())
    out = {"logits": torch.stack(logits), "image_features": f_img, "text_features": torch.stack(feats)}
    if labels is not None:
        out["loss"] = F.cross_entropy(out["logits"], labels)
    return out


def forward_backward(sd: Dict[str, torch.Tensor], image, tokenized_prompts, labels):
    sd = dict(sd)
    leaves = {}
    for k in TRAINABLE:
        leaves[k] = sd[k].detach().clone().requires_grad_(True)
        sd[k] = leaves[k]
    out = forward(sd, image, tokenized_prompts, labels)
    grads = torch.autograd.grad(out["loss"], [leaves[k] for k in TRAINABLE])
    res = {k: v.detach() for k, v in out.items()}
    res["grads"] = {k: g.detach() for k, g in zip(TRAINABLE, grads)}
    return res

"""CoCoOp on the shared native CLIP kernels -- drop-in for the reference's trainers/cocoop.py
(BASELINE config 4: instance-conditioned prompts, B x C text sequences per step).

Same public classes, constructor signatures, parameter / buffer names and return values:

  PromptLearner(cfg, classnames, clip_model) ... trainers/cocoop.py:66-163
  TextEncoder(clip_model) ...................... trainers/cocoop.py:43-64
  CustomCLIP(cfg, classnames, clip_model) ...... trainers/cocoop.py:166-198
  CoCoOp (trainer) ............................. trainers/cocoop.py:201-320

What changed underneath: the plain (cfg=None) CLIP towers run in libmudpt_b200.so; the reference's
Python loop over the images of a batch (one text-tower pass of C sequences per image, :187-192)
is ONE native text-tower call over all B x C sequences, truncated to max(eot)+1 tokens (exact under
the causal mask); the vision tower is forward-only (it holds nothing trainable).  The meta-net, the
prompt assembly and the per-image cosine logits (B x C x e multiply-adds) stay in torch autograd,
which delivers the gradients of the 5 trainable tensors from the dense d(prompts) the native text
backward returns.
"""
from __future__ import annotations

from collections import OrderedDict

import torch
from torch import nn

from .. import clip
from ..engine import text_lengths, text_tower_dense
from .mudpt import (TRAINER_REGISTRY, TrainerX, apply_freeze_rule, build_lr_scheduler, build_optimizer, load_pretrained_weights,
                    restore_checkpoints)


def load_clip_to_cpu(cfg=None):
    """trainers/cocoop.py:22-40: a plain CLIP (no cfg -> plain blocks).  Without BACKBONE.PATH the model
    is random-initialised (no checkpoint exists on the build / GPU boxes)."""
    backbone = cfg.MODEL.BACKBONE
    weights_file = getattr(backbone, "PATH", "")
    if not weights_file:
        from ..synthetic import ARCHS
        return clip.CLIP(*ARCHS[backbone.NAME].astuple(), None).float().eval()
    try:  # a TorchScript archive (the published CLIP files) ...
        weights = torch.jit.load(weights_file, map_location="cpu").state_dict()
    except RuntimeError:  # ... or a plain state dict
        weights = torch.load(weights_file, map_location="cpu")
    return clip.build_model(weights)


class TextEncoder(nn.Module):
    """trainers/cocoop.py:43-64.  The members are the CLIP's own (shared, not copied); the forward runs natively."""

    SHARED = ("transformer", "positional_embedding", "ln_final", "text_projection")

    def __init__(self, clip_model):
        super().__init__()
        for member in self.SHARED:  # (nn.Module.__setattr__ registers modules / parameters under the reference's names)
            setattr(self, member, getattr(clip_model, member))
        self.dtype = clip_model.dtype
        object.__setattr__(self, "_clip_ref", [clip_model])
        self.truncate_to_eot = True  # True / False / "per_class" (see engine.text_lengths)

    def forward(self, prompts, tokenized_prompts):
        """prompts [N, 77, d] (N = C, or B*C batched), tokenized_prompts [N, 77] -> text features [N, e]."""
        engine = self._clip_ref[0].engine(prompts.device)
        eot = tokenized_prompts.argmax(dim=-1).cpu()
        seq_len, lengths = text_lengths(eot, self.truncate_to_eot, prompts.shape[1], 1 + engine.n_ctx)
        deep = torch.zeros(0, 0, prompts.shape[-1], device=prompts.device)
        return text_tower_dense(engine, prompts.float(), eot, deep, seq_len, lengths)


class PromptLearner(nn.Module):
    """trainers/cocoop.py:66-163: context vectors `ctx` [n_ctx, d] shifted per image by `meta_net(image features)`, between
    the frozen SOS embedding (`token_prefix`) and the class-name / EOS embeddings (`token_suffix`).  Parameters are created
    in the reference's order (ctx, meta_net.linear1, meta_net.linear2), so a seeded construction draws the same values."""

    def __init__(self, cfg, classnames, clip_model, tokenizer=None, name_len=None):
        super().__init__()
        tokenize = tokenizer if tokenizer is not None else clip.tokenize
        opts = cfg.TRAINER.COCOOP
        width = clip_model.ln_final.weight.shape[0]
        feat = clip_model.visual.output_dim
        want, have = cfg.INPUT.SIZE[0], clip_model.visual.input_resolution
        assert want == have, f"cfg_imsize ({want}) must equal to clip_imsize ({have})"

        def embed(tokens):  # frozen token embedding of a tokenized batch, on whatever device the table lives
            table = clip_model.token_embedding
            with torch.no_grad():
                return table(tokens.to(table.weight.device).long()).type(clip_model.dtype)

        words = opts.CTX_INIT.replace("_", " ") if opts.CTX_INIT else ""
        if words:  # context initialised from the embedding of given words (:80-87)
            self.n_ctx = len(words.split(" "))
            start = embed(tokenize(words))[0, 1:1 + self.n_ctx, :].clone()
            lead = words
        else:  # random context N(0, 0.02^2), generic "X X ..." placeholder words (:88-92)
            self.n_ctx = opts.N_CTX
            start = torch.empty(self.n_ctx, width, dtype=clip_model.dtype)
            nn.init.normal_(start, std=0.02)
            lead = " ".join("X" for _ in range(self.n_ctx))
        self.ctx = nn.Parameter(start)
        self.meta_net = nn.Sequential(OrderedDict(
            linear1=nn.Linear(feat, feat // 16), relu=nn.ReLU(inplace=True), linear2=nn.Linear(feat // 16, width)))

        sentences = [f"{lead} {c.replace('_', ' ')}." for c in classnames]
        self.tokenized_prompts = torch.cat([tokenize(t) for t in sentences])
        fixed = embed(self.tokenized_prompts)
        self.register_buffer("token_prefix", fixed[:, :1, :].clone())                # SOS
        self.register_buffer("token_suffix", fixed[:, 1 + self.n_ctx:, :].clone())   # class name, EOS, padding
        self.n_cls = len(classnames)
        self.name_lens = name_len

    def construct_prompts(self, ctx, prefix, suffix, label=None):
        """[SOS | ctx | class tokens] along the token axis (:120-147); `label` selects classes."""
        pick = slice(None) if label is None else label
        return torch.cat([prefix[pick], ctx, suffix[pick]], dim=1)

    def forward(self, im_features):
        """[B, e] -> [B, n_cls, 77, d] (trainers/cocoop.py:149-163), built with one broadcasted cat."""
        shift = self.meta_net(im_features)                                  # [B, d]
        per_image = self.ctx.unsqueeze(0) + shift.unsqueeze(1)              # [B, n_ctx, d]
        nb = per_image.shape[0]
        return torch.cat([self.token_prefix.unsqueeze(0).expand(nb, -1, -1, -1),
                          per_image.unsqueeze(1).expand(-1, self.n_cls, -1, -1),
                          self.token_suffix.unsqueeze(0).expand(nb, -1, -1, -1)], dim=2)


class CustomCLIP(nn.Module):
    """trainers/cocoop.py:166-198."""

    def __init__(self, cfg, classnames, clip_model, tokenizer=None):
        super().__init__()
        self.prompt_learner = PromptLearner(cfg, classnames, clip_model, tokenizer=tokenizer)
        self.tokenized_prompts = self.prompt_learner.tokenized_prompts
        self.image_encoder = clip_model.visual
        self.text_encoder = TextEncoder(clip_model)
        self.logit_scale = clip_model.logit_scale
        self.dtype = clip_model.dtype
        object.__setattr__(self, "_clip_ref", [clip_model])

    def forward(self, image, label=None):
        f_img = self.image_encoder(image.type(self.dtype))
        f_img = f_img / f_img.norm(dim=-1, keepdim=True)
        prompts = self.prompt_learner(f_img)                                # [B, C, 77, d]
        nb, nc, ntok, width = prompts.shape
        # all B x C sequences in one native text-tower pass (the reference loops over the images, :187-192)
        f_txt = self.text_encoder(prompts.reshape(nb * nc, ntok, width), self.tokenized_prompts.repeat(nb, 1)).view(nb, nc, -1)
        f_txt = f_txt / f_txt.norm(dim=-1, keepdim=True)
        # per-image cosine logits: an fp32 multiply + row sum (no library GEMM, so no TF32 / algorithm dependence)
        logits = self.logit_scale.exp() * (f_img.unsqueeze(1) * f_txt).sum(dim=-1)
        if label is not None and self.prompt_learner.training:
            return nn.functional.cross_entropy(logits, label)
        return logits


@TRAINER_REGISTRY.register()
class CoCoOp(TrainerX):
    """trainers/cocoop.py:201-320 (Dassl trainer: same hooks, same registered model name, same checkpoint layout)."""

    def check_cfg(self, cfg):
        assert cfg.TRAINER.COCOOP.PREC in ["fp16", "fp32", "amp"]

    def build_model(self):
        cfg = self.cfg
        classnames = self.dm.dataset.classnames if hasattr(self, "dm") else self._classnames
        print(f"Loading CLIP (backbone: {cfg.MODEL.BACKBONE.NAME})")
        clip_model = load_clip_to_cpu(cfg).float()
        print("Building custom CLIP")
        self.model = CustomCLIP(cfg, classnames, clip_model)
        print("Turning off gradients in both the image and the text encoder")
        print(f"Parameters to be updated: {apply_freeze_rule(self.model, ('prompt_learner',))}")
        learner = self.model.prompt_learner
        if getattr(cfg.MODEL, "INIT_WEIGHTS", ""):
            load_pretrained_weights(learner, cfg.MODEL.INIT_WEIGHTS)
        self.model.to(self.device)
        # only the prompt learner goes to the optimizer and into checkpoints (:232-236)
        self.optim = build_optimizer(learner, cfg.OPTIM)
        self.sched = build_lr_scheduler(self.optim, cfg.OPTIM)
        self.register_model("prompt_learner", learner, self.optim, self.sched)
        self.scaler = None  # "amp" needs no loss scaling here: bf16 operands, fp32 accumulation and master state

    def forward_backward(self, batch):
        loss = self.model(*self.parse_batch_train(batch))
        self.optim.zero_grad()
        loss.backward()
        self.optim.step()
        if self.batch_idx + 1 == self.num_batches:
            self.update_lr()
        return {"loss": loss.item()}

    def parse_batch_train(self, batch):
        return batch["img"].to(self.device), batch["label"].to(self.device)

    def load_model(self, directory, epoch=None):
        # the fixed token vectors are recomputed from the current class names (:309-317)
        restore_checkpoints(self, directory, epoch, lambda key: key in ("token_prefix", "token_suffix"))

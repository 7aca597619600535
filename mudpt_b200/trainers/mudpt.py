"""MuDPT method plugin on the native B200 path -- drop-in for the reference's trainers/mudpt.py.

Same public classes, constructor signatures, parameter / buffer names and return shapes:

  MuDPTPromptLearner(cfg, classnames, clip_model) ... trainers/mudpt.py:41-130
  TextEncoder(clip_model) ........................... trainers/mudpt.py:133-156
  CustomCLIP(cfg, classnames, clip_model) ........... trainers/mudpt.py:159-184
  MuDPT (trainer: check_cfg / build_model / forward_backward / parse_batch_train / load_model)
                                                      trainers/mudpt.py:187-302

What changed underneath: both towers, the heads and (on the fused train path) the loss run in
libmudpt_b200.so; the class prompts are never materialised as a [C, 77, d] tensor on the fused
path (the reference's torch.cat at :106-113 is a pure copy); only the tiny [n_ctx, d] prompt
algebra (the three trainable Linear layers, :127-128 and clip/model.py:534-539) stays in torch
autograd, which is what delivers the gradients of the 10 trainable tensors.
"""
from __future__ import annotations

import math
import os
import os.path as osp
from typing import List, Optional, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import clip
from .. import dist as mdist
from ..engine import (prompt_algebra_forward, prompt_algebra_backward, text_lengths, text_tower, text_tower_dense, vision_tower, LogitsFn,
                      PromptAlgebraFn)
from ..input_pipeline import CLIP_MEAN, CLIP_STD

try:  # the Dassl engine is not in the reference tree nor in this image (SURVEY.md section 2 row 13)
    from dassl.engine import TRAINER_REGISTRY, TrainerX
    from dassl.optim import build_optimizer, build_lr_scheduler
    from dassl.utils import load_checkpoint, load_pretrained_weights
    _HAVE_DASSL = True
except Exception:  # pragma: no cover - exercised on boxes without dassl
    _HAVE_DASSL = False

    class _Registry:
        def __init__(self):
            self._m = {}

        def register(self):
            def deco(cls):
                self._m[cls.__name__] = cls
                return cls
            return deco

        def get(self, name):
            return self._m[name]

    TRAINER_REGISTRY = _Registry()

    class TrainerX:
        """Minimal stand-in for dassl.engine.TrainerX: just what `MuDPT` below touches."""

        def __init__(self, cfg=None, classnames=None, device=None):
            self.cfg = cfg
            self.device = torch.device(device) if device is not None else (
                torch.device("cuda") if torch.cuda.is_available() else torch.device("cpu"))
            self._models, self._optims, self._scheds = {}, {}, {}
            self.batch_idx, self.num_batches = 0, 1
            self._classnames = classnames
            if cfg is not None:
                self.check_cfg(cfg)
                self.build_model()

        def register_model(self, name, model, optim=None, sched=None):
            self._models[name], self._optims[name], self._scheds[name] = model, optim, sched

        def get_model_names(self):
            return list(self._models)

        def model_backward_and_update(self, loss):
            for o in self._optims.values():
                o.zero_grad()
            if not torch.isfinite(loss).all():
                raise FloatingPointError("Loss is infinite or NaN!")
            loss.backward()
            for o in self._optims.values():
                o.step()

        def update_lr(self):
            for s in self._scheds.values():
                if s is not None:
                    s.step()

        def parse_batch_test(self, batch):
            return batch["img"].to(self.device), batch["label"].to(self.device)

        def model_inference(self, input):
            return self.model(input)

        @torch.no_grad()
        def test(self, data_loader=None, split=None):
            """Dassl's TrainerX.test loop (parse_batch_test -> model_inference -> evaluator) with the Classification
            evaluator's top-1 accuracy (100 * correct / total) kept on the device: one host read for the whole split
            instead of a `.item()` per batch."""
            if data_loader is None:
                raise ValueError("the stand-in trainer has no data manager: pass the test loader")
            for m in self._models.values():
                m.eval()
            correct, total = None, 0
            for batch in data_loader:
                input, label = self.parse_batch_test(batch)
                output = self.model_inference(input)
                hits = (output.argmax(dim=1) == label).sum()
                correct = hits if correct is None else correct + hits
                total += int(label.shape[0])
            acc = 100.0 * float(correct) / max(total, 1) if correct is not None else 0.0
            self.last_test_result = {"accuracy": acc, "error_rate": 100.0 - acc, "total": total}
            return acc

        def save_model(self, epoch, directory, is_best=False, val_result=None, model_name=""):
            """Dassl's checkpoint layout (TrainerBase.save_model / dassl.utils.save_checkpoint):
            <directory>/<model name>/model.pth.tar-<epoch + 1> holding {"state_dict", "epoch", "optimizer",
            "scheduler", "val_result"} plus a "checkpoint" file naming it; `load_model` below reads it back."""
            for name in self.get_model_names():
                model = self._models[name]
                optim, sched = self._optims.get(name), self._scheds.get(name)
                fdir = osp.join(directory, name)
                os.makedirs(fdir, exist_ok=True)
                fname = model_name or ("model.pth.tar-" + str(epoch + 1))
                torch.save({"state_dict": {k: v.detach().cpu() for k, v in model.state_dict().items()}, "epoch": epoch + 1,
                            "optimizer": optim.state_dict() if optim is not None else None,
                            "scheduler": sched.state_dict() if sched is not None else None, "val_result": val_result},
                           osp.join(fdir, fname))
                with open(osp.join(fdir, "checkpoint"), "w") as f:
                    f.write(fname + "\n")
                if is_best:
                    import shutil
                    shutil.copy(osp.join(fdir, fname), osp.join(fdir, "model-best.pth.tar"))

    def build_optimizer(model, optim_cfg):
        """Dassl's SGD defaults (momentum 0.9, weight decay 5e-4); on a CUDA model the update runs as one
        native multi-tensor launch (mudpt_b200.optim.FusedSGD, same torch.optim.SGD semantics and state)."""
        params = [p for p in model.parameters() if p.requires_grad]
        kw = dict(lr=getattr(optim_cfg, "LR", 0.0025), momentum=getattr(optim_cfg, "MOMENTUM", 0.9),
                  weight_decay=getattr(optim_cfg, "WEIGHT_DECAY", 5e-4))
        if params and all(p.is_cuda for p in params) and os.environ.get("MUDPT_FUSED_SGD", "1") == "1":
            from ..optim import FusedSGD
            return FusedSGD(params, **kw)
        return torch.optim.SGD(params, **kw)

    def build_lr_scheduler(optim, optim_cfg):
        return torch.optim.lr_scheduler.CosineAnnealingLR(optim, float(getattr(optim_cfg, "MAX_EPOCH", 10)))

    def load_checkpoint(path):
        return torch.load(path, map_location="cpu", weights_only=False)

    def load_pretrained_weights(model, path):
        model.load_state_dict(load_checkpoint(path)["state_dict"], strict=False)


def load_clip_to_cpu(cfg):
    """trainers/mudpt.py:20-38.  With a BACKBONE.PATH the checkpoint's state dict is used; without one
    (no CLIP checkpoint exists on the build / GPU boxes) the model is random-initialised."""
    path = getattr(cfg.MODEL.BACKBONE, "PATH", "")
    if path:
        print(f"Loading CLIP backbone: {cfg.MODEL.BACKBONE.NAME} from {path}")
        try:
            sd = torch.jit.load(path, map_location="cpu").state_dict()
        except RuntimeError:
            sd = torch.load(path, map_location="cpu")
        return clip.build_model(sd, cfg=cfg)
    from ..synthetic import ARCHS
    print(f"No backbone path given: random-init {cfg.MODEL.BACKBONE.NAME}")
    return clip.CLIP(*ARCHS[cfg.MODEL.BACKBONE.NAME].astuple(), cfg).float().eval()


class MuDPTPromptLearner(nn.Module):
    def __init__(self, cfg, classnames, clip_model, tokenizer=None):
        super().__init__()
        tokenize = tokenizer if tokenizer is not None else clip.tokenize
        n_cls = len(classnames)
        n_ctx = cfg.TRAINER.MUDPT.N_CTX
        ctx_init = cfg.TRAINER.MUDPT.CTX_INIT
        dtype = clip_model.dtype
        ctx_dim = clip_model.ln_final.weight.shape[0]
        clip_imsize = clip_model.visual.input_resolution
        cfg_imsize = cfg.INPUT.SIZE[0]

        assert cfg.TRAINER.MUDPT.DEEP_PROMPT_DEPTH > 0, "PROMPT_DEPTH should be > 0"
        self.deep_prompts_depth = cfg.TRAINER.MUDPT.DEEP_PROMPT_DEPTH
        assert cfg_imsize == clip_imsize, f"cfg_imsize ({cfg_imsize}) must equal to clip_imsize ({clip_imsize})"

        if ctx_init:
            ctx_init = ctx_init.replace("_", " ")
            prompt = tokenize(ctx_init)
            with torch.no_grad():
                embedding = clip_model.token_embedding(prompt.to(clip_model.token_embedding.weight.device).long()).type(dtype)
            ctx_vectors = embedding[0, 1: 1 + n_ctx, :].clone()
            prompt_prefix = " ".join(ctx_init.split()[:n_ctx])
        else:
            ctx_vectors = torch.empty(n_ctx, ctx_dim, dtype=dtype)
            nn.init.normal_(ctx_vectors, std=0.02)
            prompt_prefix = " ".join(["X"] * n_ctx)
        self.ctx = nn.Parameter(ctx_vectors)

        self.embed_projection = nn.Linear(in_features=ctx_dim, out_features=clip_model.visual.positional_embedding.shape[1])
        self.deep_prompts = nn.Parameter(torch.empty(self.deep_prompts_depth - 1, n_ctx, ctx_dim))
        nn.init.normal_(self.deep_prompts, std=0.02)
        self.deep_projections = nn.Linear(ctx_dim, clip_model.visual.proj.shape[0])

        classnames = [name.replace("_", " ") for name in classnames]
        prompts = [prompt_prefix + " " + name + "." for name in classnames]
        tokenized_prompts = torch.cat([tokenize(p) for p in prompts], dim=0)  # (n_cls, 77)
        with torch.no_grad():
            embedding = clip_model.token_embedding(
                tokenized_prompts.to(clip_model.token_embedding.weight.device).long()).type(dtype)

        self.register_buffer("token_prefix", embedding[:, :1, :].clone())          # SOS
        self.register_buffer("token_suffix", embedding[:, 1 + n_ctx:, :].clone())  # CLS . EOS ~

        self.n_cls = n_cls
        self.n_ctx = n_ctx
        self.ctx_dim = ctx_dim
        self.tokenized_prompts = tokenized_prompts  # plain attribute, as in the reference (:95)

    def construct_prompts(self, ctx, prefix, suffix, label=None):
        if label is not None:
            prefix = prefix[label]
            suffix = suffix[label]
        return torch.cat([prefix, ctx, suffix], dim=1)

    def forward(self):
        """Reference API (trainers/mudpt.py:117-130): materialises the class prompts.  The fused
        CustomCLIP path does not call this."""
        ctx = self.ctx
        if ctx.dim() == 2:
            ctx = ctx.unsqueeze(0).expand(self.n_cls, self.n_ctx, self.ctx_dim)
        prompts = self.construct_prompts(ctx, self.token_prefix, self.token_suffix)
        visual_prompts = self.deep_projections(self.deep_prompts)
        t2v_shared_ctx = self.embed_projection(self.ctx.unsqueeze(0))
        return prompts, t2v_shared_ctx, self.deep_prompts, visual_prompts


class TextEncoder(nn.Module):
    def __init__(self, clip_model):
        super().__init__()
        self.transformer = clip_model.transformer
        self.positional_embedding = clip_model.positional_embedding
        self.ln_final = clip_model.ln_final
        self.text_projection = clip_model.text_projection
        self.dtype = clip_model.dtype
        # strong reference that is NOT a registered submodule (state-dict keys must match the reference)
        object.__setattr__(self, "_clip_ref", [clip_model])
        self.truncate_to_eot = True  # True / False / "per_class" (see engine.text_lengths)

    def forward(self, prompts, tokenized_prompts, deep_prompts):
        """Reference API (trainers/mudpt.py:142-156): prompts [C, 77, d] -> text features [C, e]."""
        engine = self._clip_ref[0].engine(prompts.device)
        eot = tokenized_prompts.argmax(dim=-1).cpu()
        seq_len, lengths = text_lengths(eot, self.truncate_to_eot, prompts.shape[1], 1 + engine.n_ctx)
        return text_tower_dense(engine, prompts.float(), eot, deep_prompts.float(), seq_len, lengths)


class LinfPGD:
    """l-inf PGD in pixel space against fixed text features, with the model doing the normalisation (TeCoA / APT-style
    adversarial prompt tuning and evaluation).  x_adv starts at the clean pixels (or, with random_start, at
    clamp(pixels + U(-eps, eps), 0, 1) drawn from `generator`); each step is one training vision forward on
    x_norm = (x_adv - mean) / std, the logits head (mean cross-entropy over the batch, no text-feature gradient) and
    Engine.vision_pgd_step, which updates x_adv and x_norm in place.  The start and its normalisation are PyTorch ops,
    the steps native; together they are bitwise the PyTorch loop of INTEGRATION.md."""

    def __init__(self, eng, eps, alpha, steps, random_start=False, generator=None, mean=CLIP_MEAN, std=CLIP_STD):
        if not hasattr(eng, "vision_pgd_step"):
            raise RuntimeError(f"mudpt_b200: the engine ({type(eng).__name__}) has no vision_pgd_step: it cannot run the "
                               "fused PGD attack")
        if int(steps) != steps or steps < 0:
            raise ValueError(f"mudpt_b200: PGD steps must be an integer >= 0, not {steps!r}")
        if not (math.isfinite(eps) and eps >= 0):
            raise ValueError(f"mudpt_b200: PGD eps must be finite and >= 0, not {eps!r}")
        if not (math.isfinite(alpha) and alpha > 0):
            raise ValueError(f"mudpt_b200: PGD alpha must be finite and > 0, not {alpha!r}")
        # per-channel constants as fp32 values, read once (a CUDA tensor is synchronised here, not at every step)
        self.mean, self.std = (tuple(torch.as_tensor(v, dtype=torch.float32).detach().cpu().flatten().tolist())
                               for v in (mean, std))
        if len(self.mean) != 3 or len(self.std) != 3 or not all(math.isfinite(v) and v > 0 for v in self.std):
            raise ValueError("mudpt_b200: PGD mean / std must hold 3 values each, std finite and > 0")
        self.eng, self.eps, self.alpha, self.steps = eng, float(eps), float(alpha), int(steps)
        self.random_start, self.generator = random_start, generator
        self.x_clean = self.x_adv = self.x_norm = self.label = None

    def start(self, pixels, label):
        """x_adv at the start, and x_norm = (x_adv - mean) / std (returned): PyTorch ops on the current stream"""
        self.x_clean, self.label = pixels, label.to(device=pixels.device)
        if self.random_start:
            noise = torch.empty_like(pixels).uniform_(-self.eps, self.eps, generator=self.generator)
            self.x_adv = (pixels + noise).clamp(0, 1)
        else:
            self.x_adv = pixels.clone()
        mean, std = _channel_view(self.mean, pixels.device), _channel_view(self.std, pixels.device)
        self.x_norm = (self.x_adv - mean) / std
        return self.x_norm

    def run(self, P_v, f_txt, f_img=None, forward_last=False):
        """The steps against f_txt.  f_img: the training forward of the current x_norm if already run.  With forward_last
        the result is the training forward of the final x_norm (its activations stay for a backward), else None."""
        eng, B = self.eng, self.x_adv.shape[0]
        for _ in range(self.steps):
            if f_img is None:
                f_img = eng.vision_forward(self.x_norm, P_v)
            _, _, d_i, _ = eng.logits_head(f_img, f_txt, self.label, 1.0 / B, True, text_grad=False)
            eng.vision_pgd_step(d_i, self.x_adv, self.x_clean, self.x_norm, self.mean, self.std, self.eps, self.alpha)
            f_img = None
        if forward_last and f_img is None:
            f_img = eng.vision_forward(self.x_norm, P_v)
        return f_img if forward_last else None


_CHANNEL_VIEWS = {}


def _channel_view(vals, device):
    """[1, 3, 1, 1] fp32 tensor of 3 per-channel values on `device`, cached: the host-to-device copy happens once"""
    key = (vals, str(device))
    t = _CHANNEL_VIEWS.get(key)
    if t is None:
        t = _CHANNEL_VIEWS[key] = torch.tensor(vals, dtype=torch.float32, device=device).view(1, 3, 1, 1)
    return t


class CustomCLIP(nn.Module):
    def __init__(self, cfg, classnames, clip_model, tokenizer=None):
        super().__init__()
        self.mudpt_prompt_learner = MuDPTPromptLearner(cfg, classnames, clip_model, tokenizer=tokenizer)
        self.tokenized_prompts = self.mudpt_prompt_learner.tokenized_prompts
        self.text_encoder = TextEncoder(clip_model)
        self.image_encoder = clip_model.visual
        self.logit_scale = clip_model.logit_scale
        self.dtype = clip_model.dtype
        self.deep_prompts_depth = self.mudpt_prompt_learner.deep_prompts_depth
        # strong reference that is NOT a registered submodule (state-dict keys must match the reference)
        object.__setattr__(self, "_clip_ref", [clip_model])
        # exact under the causal mask (SURVEY.md 8c-i); set False to run all 77 positions, "per_class" to run every class
        # at its own length (packed rows: no class pays for the longest one; see engine.text_lengths)
        self.truncate_text_to_eot = os.environ.get("MUDPT_TEXT_FULL_LENGTH", "0") != "1"
        self.shard_classes = True           # class-sharded text tower when torch.distributed is initialised
        self._cached_text_features = None   # eval-time cache (parameters frozen under no_grad)
        self._replicas_synced = False       # trainable tensors broadcast from rank 0 once (replicated state)
        # fused train step: vision tower on a side stream next to the text tower (see forward_backward)
        self.overlap_towers = os.environ.get("MUDPT_OVERLAP_TOWERS", "1") != "0"
        self._loss_host, self._loss_event, self._loss_pending = None, None, False

    # ------------------------------------------------------------------ helpers
    def _engine(self, device):
        return self._clip_ref[0].engine(device)

    def invalidate_cache(self):
        """Drop the evaluation-time text-feature cache (and the class set resident in the native text tower):
        call after anything that changes parameters outside forward_backward (load_state_dict, a manual update)."""
        self._cached_text_features = None
        eng = getattr(self._clip_ref[0], "_engine", None)
        if eng is not None:
            eng.class_key = None

    def _class_range(self) -> Tuple[int, int]:
        n = self.mudpt_prompt_learner.n_cls
        if self.shard_classes and mdist.world_size() > 1:
            return mdist.shard_bounds(n, mdist.rank(), mdist.world_size())
        return 0, n

    def _register_classes(self, device):
        pl = self.mudpt_prompt_learner
        if self.shard_classes and mdist.world_size() > 1 and not self._replicas_synced:
            # the prompt tensors are replicated: start every rank from rank 0's values (as DDP does)
            mdist.broadcast_params([p for p in self.parameters() if p.requires_grad])
            self._replicas_synced = True
        lo, hi = self._class_range()
        eot_all = self.tokenized_prompts.argmax(dim=-1)
        mode = self.truncate_text_to_eot
        # padded: one global length so that every rank runs the same shapes; "per_class": each shard packs its own classes
        seq_len, lengths = text_lengths(eot_all[lo:hi] if mode == "per_class" else eot_all, mode, self.tokenized_prompts.shape[1],
                                        1 + pl.n_ctx)
        eng = self._engine(device)
        key = (id(self), lo, hi, seq_len, mode)
        if eng.class_key == key:
            return
        prefix, suffix = pl.token_prefix[lo:hi], pl.token_suffix[lo:hi]
        emb = torch.cat([prefix, torch.zeros(hi - lo, pl.n_ctx, pl.ctx_dim, device=prefix.device, dtype=prefix.dtype), suffix], dim=1)
        if lengths is None:  # (engine stand-ins without the ragged form take three arguments)
            eng.text_set_classes(emb.float(), eot_all[lo:hi], seq_len)
        else:
            eng.text_set_classes(emb.float(), eot_all[lo:hi], seq_len, lengths)
        eng.class_key = key

    def _native_prompt_args(self):
        """(frozen inputs, the 10 trainable tensors in engine.PROMPT_NAMES order) of the native prompt algebra, or None
        where it does not apply (variants with extra mixing layers, CPU stand-in engine, no deep prompts)."""
        pl, ve = self.mudpt_prompt_learner, self.image_encoder
        if not (type(self) is CustomCLIP and pl.ctx.is_cuda and pl.ctx.dtype == torch.float32 and pl.deep_prompts.shape[0] > 0
                and os.environ.get("MUDPT_NATIVE_PROMPTS", "1") == "1"):
            return None
        frozen = (ve.ln_pre.eps, ve.ln_pre.weight, ve.ln_pre.bias, self.text_encoder.positional_embedding[1:1 + pl.n_ctx])
        train = [pl.ctx, pl.deep_prompts, pl.embed_projection.weight, pl.embed_projection.bias, pl.deep_projections.weight,
                 pl.deep_projections.bias, ve.visual_ctx, ve.visual_ctx_deep_prompts, ve.visual_ctx_deep_projections.weight,
                 ve.visual_ctx_deep_projections.bias]
        return frozen, train

    def prompt_stacks(self):
        """The two [depth, n_ctx, width] prompt stacks the towers splice in, as differentiable
        functions of the 10 trainable tensors (trainers/mudpt.py:127-128, :175; clip/model.py:534-539)."""
        pl, ve = self.mudpt_prompt_learner, self.image_encoder
        native = self._native_prompt_args()
        if native is not None:
            # the same algebra as below in 2 (+2 backward) native launches
            from .. import _lib
            return PromptAlgebraFn.apply(_lib.load(), *native[0], *native[1])
        visual_prompts = pl.deep_projections(pl.deep_prompts)                 # t2v deep
        shared_ctx = pl.embed_projection(pl.ctx.unsqueeze(0))                 # t2v shallow
        P_v = ve.prompt_stack(shared_ctx, visual_prompts)
        v2t = ve.visual_ctx_deep_projections(ve.visual_ctx_deep_prompts)      # v2t deep
        text_deep = pl.deep_prompts + v2t
        pos = self.text_encoder.positional_embedding[1:1 + pl.n_ctx]
        P_t = torch.cat([(pl.ctx + pos).unsqueeze(0), text_deep], dim=0).float()
        return P_v, P_t

    # ------------------------------------------------------------------ reference API
    def forward(self, image):
        """image [B, 3, H, W] -> logits [B, C] (trainers/mudpt.py:170-184), differentiable w.r.t. the prompts."""
        device = image.device
        eng = self._engine(device)
        if self.training or torch.is_grad_enabled():
            self._cached_text_features = None  # an optimizer step may follow: evaluation must recompute the text features
        self._register_classes(device)
        P_v, P_t = self.prompt_stacks()
        image_features = vision_tower(eng, image.type(self.dtype), P_v)
        text_features = text_tower(eng, P_t)
        if self.shard_classes and mdist.world_size() > 1:
            text_features = mdist.AllGatherRows.apply(text_features, self.mudpt_prompt_learner.n_cls)
        return LogitsFn.apply(eng, image_features, text_features)

    # ------------------------------------------------------------------ fused train / eval paths
    def forward_backward(self, image, label):
        """Fused train step: forward, mean cross-entropy over the GLOBAL batch (F.cross_entropy of
        trainers/mudpt.py:250 under nn.DataParallel semantics) and backward into the .grad of the 10
        trainable tensors.  Returns (loss, logits).  Gradients are all-reduced across ranks."""
        return self._fused_step(image, label, None)

    def forward_backward_adversarial(self, pixels, label, eps, alpha, steps, random_start=False, generator=None,
                                     mean=CLIP_MEAN, std=CLIP_STD):
        """Fused adversarial train step (PGD-AT / TeCoA-style adversarial prompt tuning) on pixel-space images
        `pixels` [B, 3, H, W] in [0, 1]; the model normalises with `mean` / `std`.  Returns (loss, logits, x_adv).

        One text training forward (and its all-gather across ranks), then `steps` l-inf PGD steps of size `alpha` in the
        eps-ball of `pixels` against those text features (see LinfPGD; each rank attacks its own images against all
        classes), then forward_backward's step on (x_adv - mean) / std.  Bitwise cache_text_features() + pgd_attack() +
        forward_backward(x_adv_norm), with one text forward instead of two.  The attack touches neither the text
        tower's saved activations nor any collective; with overlap_towers it runs on the vision stream."""
        device = self.logit_scale.device if pixels.device.type == "cpu" and self.logit_scale.device.type == "cuda" else pixels.device
        attack = LinfPGD(self._engine(device), eps, alpha, steps, random_start, generator, mean, std)
        loss, logits = self._fused_step(pixels, label, attack)
        return loss, logits, attack.x_adv

    def _fused_step(self, image, label, attack):
        """forward_backward, and with `attack` (a LinfPGD) forward_backward_adversarial: `image` holds the pixels, the
        vision tower's first forward is the attack's, and the attack runs between the text features and the head."""
        host_batch = image.device.type == "cpu" and self.logit_scale.device.type == "cuda"
        device = self.logit_scale.device if host_batch else image.device
        eng = self._engine(device)
        self._register_classes(device)
        self._cached_text_features = None  # the parameters are about to change: evaluation recomputes them
        world = mdist.world_size() if self.shard_classes else 1
        # Native prompt algebra without autograd when the trainable set is exactly its 10 tensors and none of them
        # carries a gradient yet (the trainer zeroes them to None): the backward kernels write straight into one flat
        # bucket whose views become the .grad tensors, and that bucket is what the ranks all-reduce.
        native = self._native_prompt_args()
        trainable = [p for p in self.parameters() if p.requires_grad]
        direct = (native is not None and len(trainable) == len(native[1]) and {id(p) for p in trainable} == {id(p) for p in native[1]}
                  and all(p.grad is None for p in trainable))
        if direct:
            from .. import _lib
            P_v, P_t, prompt_saved = prompt_algebra_forward(_lib.load(), *native[0], native[1])
        else:
            P_v, P_t = self.prompt_stacks()
        n_cls = self.mudpt_prompt_learner.n_cls
        if host_batch and not self.overlap_towers:
            image, label = image.to(device), label.to(device)
            host_batch = False
        if not host_batch:
            image = image.type(self.dtype)

        def vision_first(image, label):
            """the training vision forward that can start before the text features exist"""
            if attack is not None:
                image = attack.start(image, label)
            return eng.vision_forward(image, P_v.detach())

        if not self.overlap_towers or device.type != "cuda":  # (CPU: only the gloo tests' stand-in engine)
            f_img = vision_first(image, label)
            f_txt_loc = eng.text_forward(P_t.detach(), True)
            f_txt = mdist.all_gather_rows(f_txt_loc, n_cls) if world > 1 else f_txt_loc
            if attack is not None:
                f_img = attack.run(P_v.detach(), f_txt, f_img, forward_last=True)
            logits, loss, d_i, d_t = eng.logits_head(f_img, f_txt, label, 1.0 / (image.shape[0] * world), True)
            loss = self._publish_loss(loss, world)
            d_t_loc = mdist.reduce_scatter_rows(d_t, n_cls) if world > 1 else d_t
            dP_t, _ = eng.text_backward(d_t_loc)
            dP_v = eng.vision_backward(d_i)
        else:
            # The two towers are independent between the prompt algebra and the logits head (and again
            # after it), so the vision tower runs on a side stream next to the text tower: the tail
            # wave of one tower's persistent GEMM (e.g. 75 pair tiles on 74 SM pairs) and its small
            # latency-bound kernels are filled by the other tower's CTAs, and the text-feature
            # all-gather / reduce-scatter hide behind the vision tower.
            main = torch.cuda.current_stream(device)
            side = eng.side_stream()
            tl = self.__dict__.get("_timeline")  # diagnostic (tests/gpu_step_timeline.py): timed events at the phase boundaries

            def mark(name, stream):
                if tl is not None:
                    ev = torch.cuda.Event(enable_timing=True)
                    ev.record(stream)
                    tl.append((name, ev))

            mark("start", main)
            side.wait_stream(main)  # P_v, image are ready
            with torch.cuda.stream(side):
                if host_batch:
                    # host (pinned) batch: the upload runs on the vision stream, so the text tower -- which does
                    # not need the images -- starts at once and hides the PCIe copy (19 MB, ~0.8 ms)
                    image = image.to(device, non_blocking=True).type(self.dtype)
                    label = label.to(device, non_blocking=True)
                f_img = vision_first(image, label)
            mark("vision_fwd_end", side)
            # the head's exchange: over NVLink peer memory with the library's own kernels where the ranks share a node,
            # else NCCL collectives
            px = mdist.peer_exchange(self.__dict__, n_cls, eng.arch["embed_dim"], device) if world > 1 else None
            if px is not None:
                slot = px.next_slot()
                eng.text_forward(P_t.detach(), True, out=px.shard_out(slot))
                f_txt = px.all_gather(slot)
            else:
                f_txt_loc = eng.text_forward(P_t.detach(), True)
                f_txt = mdist.all_gather_rows(f_txt_loc, n_cls) if world > 1 else f_txt_loc
            mark("text_fwd_end", main)
            if attack is not None:
                # the attack's heads need the text features; every head of the step stays stream-ordered (one head
                # workspace per handle): the attack's on the vision stream, then the step's on the main stream
                side.wait_stream(main)
                with torch.cuda.stream(side):
                    f_img = attack.run(P_v.detach(), f_txt, f_img, forward_last=True)
                mark("attack_end", side)
            main.wait_stream(side)
            f_img.record_stream(main)
            if attack is not None:
                attack.x_adv.record_stream(main)
            if host_batch:
                label.record_stream(main)
            logits, loss, d_i, d_t = eng.logits_head(f_img, f_txt, label, 1.0 / (image.shape[0] * world), True,
                                                     d_t_out=px.grad_out(slot) if px is not None else None)
            loss = self._publish_loss(loss, world)
            mark("head_end", main)
            side.wait_stream(main)  # d_i
            with torch.cuda.stream(side):
                dP_v = eng.vision_backward(d_i)
            mark("vision_bwd_end", side)
            d_i.record_stream(side)
            if px is not None:
                d_t_loc = px.reduce_scatter(slot)
            else:
                d_t_loc = mdist.reduce_scatter_rows(d_t, n_cls) if world > 1 else d_t
            dP_t, _ = eng.text_backward(d_t_loc)
            mark("text_bwd_end", main)
            main.wait_stream(side)
            dP_v.record_stream(main)
        if direct:
            fg = self.__dict__.get("_flat_grads")
            if fg is None or not fg.matches(native[1]):
                fg = mdist.FlatGrads(native[1])
                self.__dict__["_flat_grads"] = fg
            prompt_algebra_backward(_lib.load(), prompt_saved, dP_v, dP_t, fg.views)
            for p, v in zip(fg.params, fg.views):
                p.grad = v
            if world > 1:
                fg.all_reduce()  # one collective on the bucket itself: no concatenation, no copies back
            if self.__dict__.get("_timeline") is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record(torch.cuda.current_stream(device))
                self.__dict__["_timeline"].append(("grads_end", ev))
        else:
            torch.autograd.backward([P_v, P_t], [dP_v, dP_t])
            if world > 1:
                mdist.all_reduce_grads(trainable)
        return loss, logits

    def _publish_loss(self, loss, world):
        """Global loss right after the head: all-reduce across ranks, then an asynchronous copy into pinned host
        memory + an event, so that the trainer can read the value (loss_value()) while the backward is still
        running instead of draining the stream with loss.item()."""
        if world > 1:
            loss = mdist.all_reduce_sum(loss)
        if loss.is_cuda:
            if self._loss_host is None:
                self._loss_host = torch.empty((), dtype=torch.float32).pin_memory()
                self._loss_event = torch.cuda.Event()
            self._loss_host.copy_(loss, non_blocking=True)
            self._loss_event.record(torch.cuda.current_stream(loss.device))
            self._loss_pending = True
        return loss

    def loss_value(self) -> float:
        """Python float of the last fused step's loss; waits only for the head, not for the backward."""
        if not self._loss_pending:
            raise RuntimeError("loss_value(): no fused step has been run")
        self._loss_event.synchronize()
        return float(self._loss_host)

    @torch.no_grad()
    def cache_text_features(self, device=None):
        """Text features depend only on parameters: compute them once for evaluation (the reference
        recomputes the text tower for every test batch, SURVEY.md 3.4)."""
        device = device or self.logit_scale.device
        eng = self._engine(device)
        self._register_classes(device)
        _, P_t = self.prompt_stacks()
        f = text_tower(eng, P_t)
        if self.shard_classes and mdist.world_size() > 1:
            f = mdist.all_gather_rows(f, self.mudpt_prompt_learner.n_cls)
        self._cached_text_features = f
        return f

    @torch.no_grad()
    def inference(self, image):
        """logits with cached text features (call cache_text_features() first / after each update)."""
        if self._cached_text_features is None:
            self.cache_text_features(image.device)
        eng = self._engine(image.device)
        P_v, _ = self.prompt_stacks()
        f_img = vision_tower(eng, image.type(self.dtype), P_v)
        logits, _, _, _ = eng.logits_head(f_img, self._cached_text_features, None, 1.0, False)
        return logits

    @torch.no_grad()
    def image_gradient(self, image, label):
        """Fused attack step (PGD, AutoAttack, adversarial prompt tuning): (loss, logits, d_image) of the mean
        cross-entropy over this batch w.r.t. `image` [B, 3, H, W] (the tensor as given, after pixel normalisation).

        The text features are the cached ones (computed like inference() does if there are none), so no text tower and no
        collective runs: under torchrun every rank attacks its own images.  One training vision forward with the prompts
        detached, the logits head with `label` (the text-feature gradient is not computed) and the vision backward into
        the images, without autograd.  `logits` are bitwise those of inference(image).

        The vision forward here replaces the tower's saved activations (it moves the engine's vision generation): a
        vision backward still pending from an earlier forward raises instead of returning wrong gradients."""
        if self._cached_text_features is None:
            self.cache_text_features(image.device)
        eng = self._engine(image.device)
        P_v, _ = self.prompt_stacks()
        image = image.type(self.dtype)
        f_img = eng.vision_forward(image, P_v.detach())
        logits, loss, d_i, _ = eng.logits_head(f_img, self._cached_text_features, label, 1.0 / image.shape[0], True,
                                               text_grad=False)
        _, d_image = eng.vision_backward_images(d_i, want_prompts=False)
        return loss, logits, d_image

    @torch.no_grad()
    def pgd_attack(self, pixels, label, eps, alpha, steps, random_start=False, generator=None, mean=CLIP_MEAN, std=CLIP_STD):
        """l-inf PGD on the cached text features (adversarial evaluation): `steps` steps of size `alpha` in the eps-ball of
        `pixels` [B, 3, H, W] in [0, 1], starting there or (random_start) at clamp(pixels + U(-eps, eps), 0, 1) drawn from
        `generator`.  The model normalises with `mean` / `std`.  Returns (x_adv, x_adv_norm = (x_adv - mean) / std).

        Each step is one training vision forward, the logits head (mean cross-entropy over this batch) and one native
        PGD step (Engine.vision_pgd_step): no autograd, no text tower, no collective (under torchrun every rank attacks
        its own images).  Bitwise the PyTorch loop of INTEGRATION.md on image_gradient.  As image_gradient, the vision
        forwards replace the tower's saved activations: a vision backward still pending from an earlier forward raises."""
        if self._cached_text_features is None:
            self.cache_text_features(pixels.device)
        eng = self._engine(pixels.device)
        attack = LinfPGD(eng, eps, alpha, steps, random_start, generator, mean, std)
        P_v, _ = self.prompt_stacks()
        attack.start(pixels.type(self.dtype), label)
        attack.run(P_v.detach(), self._cached_text_features)
        return attack.x_adv, attack.x_norm


@TRAINER_REGISTRY.register()
def apply_freeze_rule(model, keep):
    """The reference trainers' freeze rule (trainers/mudpt.py:205-212, trainers/cocoop.py:221-225): a parameter stays
    trainable iff its name contains one of the substrings `keep`; everything else (the whole CLIP) is frozen.
    Returns the set of trainable names."""
    for pname, p in model.named_parameters():
        p.requires_grad_(any(k in pname for k in keep))
    return {pname for pname, p in model.named_parameters() if p.requires_grad}


def restore_checkpoints(trainer, directory, epoch, is_class_bound, after_load=None):
    """Body of the reference trainers' load_model (trainers/mudpt.py:270-302, trainers/cocoop.py:285-320): for every
    registered model read Dassl's `<directory>/<name>/model-best.pth.tar` (or `model.pth.tar-<epoch>`), drop the entries
    that depend on the class names (`is_class_bound(key)`: the fixed token vectors, recomputed from the current names)
    and load the rest non-strictly.  FileNotFoundError as in the reference."""
    if not directory:
        print("Note that load_model() is skipped as no pretrained model is given")
        return
    fname = "model-best.pth.tar" if epoch is None else "model.pth.tar-" + str(epoch)
    for name in trainer.get_model_names():
        path = osp.join(directory, name, fname)
        if not osp.exists(path):
            raise FileNotFoundError('Model not found at "{}"'.format(path))
        ckpt = load_checkpoint(path)
        weights = {k: v for k, v in ckpt["state_dict"].items() if not is_class_bound(k)}
        print('Loading weights to {} from "{}" (epoch = {})'.format(name, path, ckpt["epoch"]))
        trainer._models[name].load_state_dict(weights, strict=False)
        if after_load is not None:
            after_load(trainer._models[name])


class MuDPT(TrainerX):
    def check_cfg(self, cfg):
        assert cfg.TRAINER.MUDPT.PREC in ["fp16", "fp32", "amp"]

    def build_model(self):
        cfg = self.cfg
        classnames = self.dm.dataset.classnames if hasattr(self, "dm") else self._classnames
        print(f"Loading CLIP (backbone: {cfg.MODEL.BACKBONE.NAME})")
        clip_model = load_clip_to_cpu(cfg)
        clip_model.float()  # the reference's effective numerics are fp32 for every PREC (SURVEY.md section 5)

        print("Building custom CLIP")
        self.model = CustomCLIP(cfg, classnames, clip_model)

        print("Turning off gradients in both the image and the text encoder")
        enabled = apply_freeze_rule(self.model, ("prompt_learner", "visual_ctx"))
        print(f"Parameters to be updated: {enabled}")

        if getattr(cfg.MODEL, "INIT_WEIGHTS", ""):
            load_pretrained_weights(self.model.mudpt_prompt_learner, cfg.MODEL.INIT_WEIGHTS)

        self.model.to(self.device)
        self.optim = build_optimizer(self.model, cfg.OPTIM)
        self.sched = build_lr_scheduler(self.optim, cfg.OPTIM)
        self.register_model("MultimodalDeepPromptTuning", self.model, self.optim, self.sched)
        self.scaler = None  # "amp" needs no loss scaling here: bf16 operands, fp32 accumulation and master state

    def prefetch(self, batch):
        """Start the host -> device copy of a FUTURE batch (what a pinned-memory data loader with non_blocking copies
        does): call it with batch i + 1 before forward_backward(batch i); the upload then runs on a copy stream under
        step i and forward_backward(batch i + 1) finds the images resident.  Two device slots, reused alternately; a slot
        is only overwritten after the step that read it has finished (event-ordered, no host synchronisation)."""
        if "img" not in batch or self.device.type != "cuda" or batch["img"].device.type != "cpu":
            return
        st = self.__dict__.setdefault("_pf", {"slot": 0, "bufs": [None, None], "free": [None, None], "ready": {}, "stream": torch.cuda.Stream(self.device)})
        k = st["slot"]
        st["slot"] ^= 1
        img, lab = batch["img"], batch["label"]
        buf = st["bufs"][k]
        if buf is None or buf[0].shape != img.shape or buf[0].dtype != img.dtype or buf[1].shape != lab.shape:
            buf = (torch.empty(img.shape, dtype=img.dtype, device=self.device), torch.empty(lab.shape, dtype=lab.dtype, device=self.device))
            st["bufs"][k] = buf
        cs = st["stream"]
        if st["free"][k] is None:
            cs.wait_stream(torch.cuda.current_stream(self.device))  # first use of the slot: its allocation is ordered there
        else:
            cs.wait_event(st["free"][k])                            # the step that read the slot last has finished
        with torch.cuda.stream(cs):
            buf[0].copy_(img, non_blocking=True)
            buf[1].copy_(lab, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(cs)
        # (a batch prefetched into this slot earlier and never consumed is forgotten: its step uploads in the call)
        st["ready"] = {key: r for key, r in st["ready"].items() if r["slot"] != k}
        st["ready"][id(img)] = {"slot": k, "event": ev, "host": img}  # (the reference keeps the id from being reused)

    def _prefetched(self, batch):
        st = self.__dict__.get("_pf")
        r = st["ready"].pop(id(batch.get("img")), None) if st else None
        if r is None:
            return None
        torch.cuda.current_stream(self.device).wait_event(r["event"])
        return r["slot"], st["bufs"][r["slot"]]

    def forward_backward(self, batch):
        if os.environ.get("MUDPT_FUSED_STEP", "1") == "1":
            # fused loss + backward in the native head; same update as model_backward_and_update(loss).
            # Host batches go in as they are: the fused step uploads them on its vision stream
            # (parse_batch_train's blocking .to(device) would put the PCIe copy on the critical path).
            pf = self._prefetched(batch) if "img" in batch else None
            if pf is not None:
                image, label = pf[1]  # uploaded by prefetch() under the previous step
            elif "img" not in batch:
                image, label = self.parse_batch_train(batch)  # raw 8-bit images: GPU input pipeline
            else:
                image, label = batch["img"], batch["label"]
                if not (image.device.type == "cpu" and self.device.type == "cuda"):
                    image, label = self.parse_batch_train(batch)
            self.optim.zero_grad()
            loss, _ = self.model.forward_backward(image, label)
            if pf is not None:  # the slot may be refilled once this step (both streams joined on the current one) is done
                ev = torch.cuda.Event()
                ev.record(torch.cuda.current_stream(self.device))
                self._pf["free"][pf[0]] = ev
            # the loss value is on the host as soon as the head has run (the backward is still in flight):
            # same check-before-update order as model_backward_and_update, without draining the stream
            loss_value = self.model.loss_value() if loss.is_cuda else float(loss)
            if not math.isfinite(loss_value):
                raise FloatingPointError("Loss is infinite or NaN!")
            self.optim.step()
            if (self.batch_idx + 1) == self.num_batches:
                self.update_lr()
            return {"loss": loss_value}
        else:
            image, label = self.parse_batch_train(batch)
            output = self.model(image)
            world = mdist.world_size() if getattr(self.model, "shard_classes", False) else 1
            loss = F.cross_entropy(output, label)
            if world > 1:
                # class-sharded text tower + data-parallel images: the update must be the GLOBAL-batch mean
                # (nn.DataParallel semantics, trainers/mudpt.py:230-233), summed over ranks before the step
                for o in self._optims.values():
                    o.zero_grad()
                (loss / world).backward()
                mdist.all_reduce_grads([p for p in self.model.parameters() if p.requires_grad])
                loss = mdist.all_reduce_sum(loss.detach()) / world
                if not torch.isfinite(loss).all():
                    raise FloatingPointError("Loss is infinite or NaN!")
                for o in self._optims.values():
                    o.step()
            else:
                self.model_backward_and_update(loss)
        loss_summary = {"loss": loss.item()}
        if (self.batch_idx + 1) == self.num_batches:
            self.update_lr()
        return loss_summary

    def parse_batch_train(self, batch):
        if "img" not in batch:
            # SURVEY.md 8f N2: batch["img_u8"] = list of decoded 8-bit RGB images [H, W, 3] (any sizes, host or
            # device).  The transform the yaml names (random_resized_crop, random_flip, normalize; bicubic) runs on
            # the GPU, bit-identical to the torchvision / PIL pipeline of the reference's data loader.
            input = self.input_transform()(batch["img_u8"])
            return input, batch["label"].to(self.device)
        input = batch["img"].to(self.device)
        label = batch["label"].to(self.device)
        return input, label

    def parse_batch_test(self, batch):
        """Dassl TrainerX.parse_batch_test; raw 8-bit images go through the evaluation transform
        (Resize(max(size)) -> CenterCrop -> normalize) on the GPU."""
        if "img" not in batch:
            return self.input_transform(False)(batch["img_u8"]), batch["label"].to(self.device)
        return batch["img"].to(self.device), batch["label"].to(self.device)

    def model_inference(self, input):
        """Dassl TrainerX.model_inference (`self.model(input)` in the reference, which recomputes the text tower for
        every test batch): the text features depend only on parameters, so they are computed once per evaluation
        (SURVEY.md 8f N1) -- the cache is dropped by every training step."""
        return self.model.inference(input)

    def input_transform(self, is_train: bool = True):
        """GpuTransform built from cfg.INPUT (mudpt_b200/input_pipeline.py), one per mode, created on first use."""
        cache = self.__dict__.setdefault("_input_transforms", {})
        if is_train not in cache:
            from ..input_pipeline import GpuTransform
            cache[is_train] = GpuTransform.from_cfg(self.cfg, is_train, device=self.device)
        return cache[is_train]

    def load_model(self, directory, epoch=None):
        # class names may differ (base -> new): ignore the fixed token vectors, whatever the learner is called
        # (mudpt_ / umudpt_ / uumudpt_prompt_learner: trainers/mudpt.py:294-298, umudpt.py:337-341, uumudpt.py:343-347)
        def token_vector(key):
            return key.endswith(("prompt_learner.token_prefix", "prompt_learner.token_suffix"))

        def refresh(model):
            model._clip_ref[0].refresh_engine_weights()
            model.invalidate_cache()  # cached text features / resident class set belong to the old weights

        restore_checkpoints(self, directory, epoch, token_vector, refresh)

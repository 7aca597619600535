"""TEST INFRASTRUCTURE ONLY -- import the read-only reference under import shims.

The reference (a checkout of the original MuDPT Python project, not part of this repository,
located by the environment variable MUDPT_REFERENCE_ROOT) needs `yacs`, `dassl` and `ftfy`
(SURVEY.md section 8c).  This module registers minimal stand-ins *before*
importing the reference packages so that the reference's own `clip/model.py` and
`trainers/mudpt.py` run unmodified on CPU fp32.  It is used only

  * by `oracle/make_golden.py` to generate the golden fixtures committed under tests/golden/, and
  * by tests marked `needs_reference` that pin the restatement in `oracle/mudpt_oracle.py`
    against the reference itself.

Nothing under mudpt_b200/ imports this file.  `reference_available()` is the gate: without
MUDPT_REFERENCE_ROOT the golden fixtures stand in for the reference.
"""
from __future__ import annotations

import os
import sys
import types

REFERENCE_ROOT = os.environ.get("MUDPT_REFERENCE_ROOT", "")


def reference_available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isfile(os.path.join(REFERENCE_ROOT, "trainers", "mudpt.py"))


class CfgNode(dict):
    """Attribute-access dict; enough for the reference, which only reads cfg values
    (clip/model.py:268,510-511; trainers/mudpt.py:44-55)."""

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:  # pragma: no cover
            raise AttributeError(k) from e

    def __setattr__(self, k, v):
        self[k] = v


def make_cfg(n_ctx: int = 2, depth: int = 9, ctx_init: str = "a photo of a",
             prec: str = "fp32", size: int = 224, name: str = "MuDPT") -> CfgNode:
    """The subset of the yacs tree the hot path reads (train.py:114-119)."""
    cfg = CfgNode()
    cfg.TRAINER = CfgNode()
    cfg.TRAINER.NAME = name
    cfg.TRAINER.MUDPT = CfgNode(N_CTX=n_ctx, CTX_INIT=ctx_init, DEEP_PROMPT_DEPTH=depth, PREC=prec)
    cfg.TRAINER.COCOOP = CfgNode(N_CTX=n_ctx, CTX_INIT=ctx_init, PREC=prec)  # trainers/cocoop.py:69-70
    cfg.TRAINER.UMUDPT = CfgNode(N_CTX=n_ctx, CTX_INIT=ctx_init, DEEP_PROMPT_DEPTH=depth, PREC=prec)
    cfg.TRAINER.UUMUDPT = CfgNode(N_CTX=n_ctx, CTX_INIT=ctx_init, DEEP_PROMPT_DEPTH=depth, PREC=prec)
    cfg.INPUT = CfgNode(SIZE=(size, size))
    cfg.MODEL = CfgNode(BACKBONE=CfgNode(NAME="ViT-B/16", PATH=""), INIT_WEIGHTS="")
    return cfg


def _install_shims() -> None:
    if "yacs" not in sys.modules:
        yacs = types.ModuleType("yacs")
        yacs_config = types.ModuleType("yacs.config")
        yacs_config.CfgNode = CfgNode
        yacs.config = yacs_config
        sys.modules["yacs"] = yacs
        sys.modules["yacs.config"] = yacs_config
    if "ftfy" not in sys.modules:
        ftfy = types.ModuleType("ftfy")
        ftfy.fix_text = lambda s: s  # identity is exact for ASCII class names
        sys.modules["ftfy"] = ftfy
    if "dassl" not in sys.modules:
        dassl = types.ModuleType("dassl")

        class _Registry:
            def register(self, *a, **k):
                return lambda cls: cls

        class TrainerX:  # empty base; the trainer loop is out of scope
            pass

        def _nope(*a, **k):  # pragma: no cover
            raise NotImplementedError("dassl is not in the tree (SURVEY.md section 2, row 13)")

        engine = types.ModuleType("dassl.engine")
        engine.TRAINER_REGISTRY = _Registry()
        engine.TrainerX = TrainerX
        metrics = types.ModuleType("dassl.metrics")
        metrics.compute_accuracy = _nope
        utils = types.ModuleType("dassl.utils")
        utils.load_pretrained_weights = _nope
        utils.load_checkpoint = _nope
        optim = types.ModuleType("dassl.optim")
        optim.build_optimizer = _nope
        optim.build_lr_scheduler = _nope
        for name, mod in [("dassl", dassl), ("dassl.engine", engine), ("dassl.metrics", metrics),
                          ("dassl.utils", utils), ("dassl.optim", optim)]:
            sys.modules[name] = mod
        dassl.engine, dassl.metrics, dassl.utils, dassl.optim = engine, metrics, utils, optim


def import_reference():
    """Returns (clip_pkg, clip.model module, trainers.mudpt module) of the reference."""
    if not reference_available():
        raise RuntimeError(f"reference not found: set MUDPT_REFERENCE_ROOT to a MuDPT checkout (now {REFERENCE_ROOT!r})")
    _install_shims()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import importlib
    clip_pkg = importlib.import_module("clip")
    clip_model = importlib.import_module("clip.model")
    ref_mudpt = importlib.import_module("trainers.mudpt")
    return clip_pkg, clip_model, ref_mudpt


def import_reference_variant(name: str):
    """The reference's trainers/umudpt.py or trainers/uumudpt.py (SURVEY 8f N4), under the same shims."""
    import importlib
    import_reference()
    return importlib.import_module("trainers." + name.lower())


def import_reference_cocoop():
    """The reference's trainers/cocoop.py (BASELINE config 4), under the same shims."""
    import importlib
    import_reference()
    return importlib.import_module("trainers.cocoop")


ARCH = {
    # embed_dim, image_resolution, vision_layers, vision_width, vision_patch_size,
    # context_length, vocab_size, transformer_width, transformer_heads, transformer_layers
    "ViT-B/16": (512, 224, 12, 768, 16, 77, 49408, 512, 8, 12),
    "ViT-B/32": (512, 224, 12, 768, 32, 77, 49408, 512, 8, 12),
    "ViT-L/14": (768, 224, 24, 1024, 14, 77, 49408, 768, 12, 12),
    # small shapes for fast CPU tests (same code path, heads of 64)
    "tiny": (128, 32, 3, 128, 16, 77, 49408, 128, 2, 3),
}


def build_reference_model(arch: str = "ViT-B/16", classnames=None, seed: int = 0,
                          n_ctx: int = 2, depth: int = 9, ctx_init: str = "a photo of a"):
    """Random-init reference CustomCLIP in fp32 with the freeze rule of
    trainers/mudpt.py:205-212 applied by hand.  Returns (model, cfg)."""
    import torch
    _, clip_model_mod, ref_mudpt = import_reference()
    a = ARCH[arch]
    cfg = make_cfg(n_ctx=n_ctx, depth=depth, ctx_init=ctx_init, size=a[1])
    torch.manual_seed(seed)
    clip_model = clip_model_mod.CLIP(*a, cfg).float()
    if classnames is None:
        classnames = [f"class {i}" for i in range(100)]
    model = ref_mudpt.CustomCLIP(cfg, classnames, clip_model)
    for name, p in model.named_parameters():
        if "prompt_learner" not in name:
            p.requires_grad_("visual_ctx" in name)
    return model, cfg

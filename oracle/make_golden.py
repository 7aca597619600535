"""TEST INFRASTRUCTURE ONLY -- generate tests/golden/*.npz from the REFERENCE itself.

Needs the reference (MUDPT_REFERENCE_ROOT, imported read-only under
oracle/ref_shims.py).  For each case it

  1. builds the reference `CLIP(...)` + `trainers.mudpt.CustomCLIP` (unmodified reference
     code, fp32 CPU),
  2. loads the deterministic synthetic weights of mudpt_b200/synthetic.py into it
     (so the fixture does not have to carry the weights),
  3. runs one forward + `F.cross_entropy` + backward exactly as
     `MuDPT.forward_backward` does (trainers/mudpt.py:249-251, minus the optimizer), and
  4. stores token ids, logits, features, loss and the 10 prompt gradients.

    python oracle/make_golden.py            # all cases
"""
from __future__ import annotations

import os
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_shims  # noqa: E402
from mudpt_b200 import synthetic as syn  # noqa: E402
from tests import golden_util as gu  # noqa: E402

CASES = {
    # name: arch, n_ctx, depth, ctx_init, classnames, batch, image kind
    "tiny_a": dict(arch="tiny", n_ctx=2, depth=2, ctx_init="a photo of a",
                   classnames=["cat", "airplane model", "class 12", "x", "very long bird name here"], batch=3, kind="noise"),
    "tiny_b": dict(arch="tiny2", n_ctx=4, depth=2, ctx_init="",
                   classnames=["class 0", "class 1", "dog", "sun flower"], batch=2, kind="noise"),
    "tiny_c": dict(arch="tiny", n_ctx=2, depth=1, ctx_init="a photo of a",
                   classnames=["class 0", "class 1", "class 2"], batch=2, kind="colour"),
    "tiny_d": dict(arch="tiny", n_ctx=3, depth=3, ctx_init="",
                   classnames=[f"class {i}" for i in range(17)], batch=5, kind="noise"),
    # BASELINE config 1: ViT-B/16, n_ctx 2, depth 9, B=4, C=100
    "vitb16_cfg1": dict(arch="ViT-B/16", n_ctx=2, depth=9, ctx_init="a photo of a",
                        classnames=[f"class {i}" for i in range(100)], batch=4, kind="noise"),
}


def run_case(name: str, spec: dict, out_dir: str) -> None:
    clip_pkg, clip_model_mod, ref_mudpt = ref_shims.import_reference()
    arch = syn.ARCHS[spec["arch"]]
    cfg = ref_shims.make_cfg(n_ctx=spec["n_ctx"], depth=spec["depth"], ctx_init=spec["ctx_init"],
                             size=arch.image_resolution)
    t0 = time.time()
    clip_model = clip_model_mod.CLIP(*arch.astuple(), cfg).float()
    clip_sd = syn.synthetic_clip_state_dict(arch, seed=0)
    pp = syn.synthetic_prompt_params(arch, spec["n_ctx"], spec["depth"], seed=0)
    full = dict(clip_sd)
    for k, v in pp.items():
        if k.startswith("visual."):
            full[k] = v
    missing, unexpected = clip_model.load_state_dict(full, strict=True), None
    model = ref_mudpt.CustomCLIP(cfg, spec["classnames"], clip_model)
    pl = model.mudpt_prompt_learner
    with torch.no_grad():
        pl.deep_prompts.copy_(pp["prompt.deep_prompts"])
        pl.embed_projection.weight.copy_(pp["prompt.embed_projection.weight"])
        pl.embed_projection.bias.copy_(pp["prompt.embed_projection.bias"])
        pl.deep_projections.weight.copy_(pp["prompt.deep_projections.weight"])
        pl.deep_projections.bias.copy_(pp["prompt.deep_projections.bias"])
        if not spec["ctx_init"]:
            pl.ctx.copy_(pp["prompt.ctx_random"])
    # freeze rule, trainers/mudpt.py:205-212
    for n, p in model.named_parameters():
        if "prompt_learner" not in n:
            p.requires_grad_("visual_ctx" in n)
    trainable = [n for n, p in model.named_parameters() if p.requires_grad]
    tokenized = model.tokenized_prompts.clone()
    ctx_tokens = clip_pkg.tokenize(spec["ctx_init"].replace("_", " "))[0] if spec["ctx_init"] else None

    # the assembled synthetic state dict must equal the reference module's own state dict
    mine = syn.assemble_state_dict(arch, tokenized, spec["n_ctx"], spec["depth"], ctx_tokens, seed=0, clip_sd=clip_sd)
    ref_sd = model.state_dict()
    assert set(mine) == set(ref_sd), (set(mine) ^ set(ref_sd))
    for k in ref_sd:
        assert torch.equal(mine[k], ref_sd[k]), k

    image = syn.synthetic_images(spec["batch"], arch.image_resolution, seed=1, kind=spec["kind"])
    labels = syn.synthetic_labels(spec["batch"], len(spec["classnames"]), seed=1)
    model.zero_grad()
    logits = model(image)                       # trainers/mudpt.py:249
    loss = F.cross_entropy(logits, labels)      # :250
    loss.backward()                             # :251 (model_backward_and_update minus optim.step)
    with torch.no_grad():
        prompts, shared, text_deep, t2v = model.mudpt_prompt_learner()
        f_img, v2t = model.image_encoder(image, shared, t2v)
        f_txt = model.text_encoder(prompts, tokenized, text_deep + v2t)
    out = {
        "arch": np.array(spec["arch"]), "n_ctx": np.array(spec["n_ctx"]), "depth": np.array(spec["depth"]),
        "batch": np.array(spec["batch"]), "kind": np.array(spec["kind"]),
        "classnames": np.array(spec["classnames"]),
        "has_ctx_init": np.array(bool(spec["ctx_init"])),
        "ctx_init_tokens": (ctx_tokens.numpy() if ctx_tokens is not None else np.zeros(0, np.int32)),
        "tokenized_prompts": tokenized.numpy().astype(np.int32),
        "labels": labels.numpy(),
        "logits": logits.detach().numpy(), "loss": loss.detach().numpy(),
        "image_features": f_img.numpy(), "text_features": f_txt.numpy(),
    }
    for n, p in model.named_parameters():
        if p.requires_grad:
            # depth == 1: the deep tensors have leading dim 0 and autograd leaves .grad None
            out["grad/" + n] = (p.grad if p.grad is not None else torch.zeros_like(p)).numpy()
    assert len(trainable) == 10, trainable
    path = os.path.join(out_dir, name + ".npz")
    gu.save(path, out)
    print(f"{name}: loss={float(loss.detach()):.6f} logits{tuple(logits.shape)} -> {path} "
          f"({os.path.getsize(path)/1e6:.2f} MB, {time.time()-t0:.1f}s)")


COCOOP_CASES = {
    # BASELINE config 4 (CoCoOp-style instance-conditioned prompts), small shapes
    "cocoop_tiny_a": dict(arch="tiny", n_ctx=4, ctx_init="a photo of a",
                          classnames=["cat", "airplane model", "class 12", "x", "very long bird name here"], batch=3, kind="noise"),
    "cocoop_tiny_b": dict(arch="tiny2", n_ctx=2, ctx_init="",
                          classnames=["class 0", "class 1", "dog", "sun flower"], batch=2, kind="colour"),
}


def run_cocoop_case(name: str, spec: dict, out_dir: str) -> None:
    """Unmodified reference trainers/cocoop.py CustomCLIP on the plain (cfg=None) reference CLIP."""
    clip_pkg, clip_model_mod, _ = ref_shims.import_reference()
    ref_cocoop = ref_shims.import_reference_cocoop()
    arch = syn.ARCHS[spec["arch"]]
    cfg = ref_shims.make_cfg(n_ctx=spec["n_ctx"], depth=1, ctx_init=spec["ctx_init"], size=arch.image_resolution, name="CoCoOp")
    t0 = time.time()
    clip_model = clip_model_mod.CLIP(*arch.astuple(), None).float()
    clip_sd = syn.synthetic_clip_state_dict(arch, seed=0)
    clip_model.load_state_dict(clip_sd, strict=True)
    model = ref_cocoop.CustomCLIP(cfg, spec["classnames"], clip_model)
    pp = syn.synthetic_cocoop_params(arch, spec["n_ctx"], seed=0)
    pl = model.prompt_learner
    with torch.no_grad():
        for k in ("linear1.weight", "linear1.bias", "linear2.weight", "linear2.bias"):
            getattr(getattr(pl.meta_net, k.split(".")[0]), k.split(".")[1]).copy_(pp["meta_net." + k])
        if not spec["ctx_init"]:
            pl.ctx.copy_(pp["ctx_random"])
    for n, p in model.named_parameters():   # freeze rule, trainers/cocoop.py:221-225
        if "prompt_learner" not in n:
            p.requires_grad_(False)
    trainable = [n for n, p in model.named_parameters() if p.requires_grad]
    assert len(trainable) == 5, trainable
    tokenized = model.tokenized_prompts.clone()
    ctx_tokens = clip_pkg.tokenize(spec["ctx_init"].replace("_", " "))[0] if spec["ctx_init"] else None
    mine = syn.assemble_cocoop_state_dict(arch, tokenized, pl.n_ctx, ctx_tokens, seed=0, clip_sd=clip_sd)
    ref_sd = model.state_dict()
    assert set(mine) == set(ref_sd), (set(mine) ^ set(ref_sd))
    for k in ref_sd:
        assert torch.equal(mine[k], ref_sd[k]), k
    image = syn.synthetic_images(spec["batch"], arch.image_resolution, seed=1, kind=spec["kind"])
    labels = syn.synthetic_labels(spec["batch"], len(spec["classnames"]), seed=1)
    model.train()
    model.zero_grad()
    loss = model(image, labels)     # trainers/cocoop.py:262 (training branch returns the cross-entropy, :195-196)
    loss.backward()
    model.eval()
    with torch.no_grad():
        logits = model(image)
    out = {
        "arch": np.array(spec["arch"]), "n_ctx": np.array(pl.n_ctx), "batch": np.array(spec["batch"]), "kind": np.array(spec["kind"]),
        "classnames": np.array(spec["classnames"]), "has_ctx_init": np.array(bool(spec["ctx_init"])),
        "ctx_init": np.array(spec["ctx_init"]),
        "ctx_init_tokens": (ctx_tokens.numpy() if ctx_tokens is not None else np.zeros(0, np.int32)),
        "tokenized_prompts": tokenized.numpy().astype(np.int32), "labels": labels.numpy(),
        "logits": logits.numpy(), "loss": loss.detach().numpy(),
    }
    for n, p in model.named_parameters():
        if p.requires_grad:
            out["grad/" + n] = p.grad.numpy()
    path = os.path.join(out_dir, name + ".npz")
    gu.save(path, out)
    print(f"{name}: loss={float(loss.detach()):.6f} logits{tuple(logits.shape)} -> {path} "
          f"({os.path.getsize(path)/1e6:.2f} MB, {time.time()-t0:.1f}s)")


VARIANT_CASES = {
    # SURVEY 8f N4: UMuDPT / UUMuDPT (LightTransformer-mixed prompts on the same towers)
    "umudpt_tiny": dict(trainer="UMuDPT", arch="tiny", n_ctx=2, depth=3, ctx_init="a photo of a",
                        classnames=["cat", "airplane model", "class 12", "x"], batch=3, kind="noise"),
    "uumudpt_tiny": dict(trainer="UUMuDPT", arch="tiny", n_ctx=3, depth=2, ctx_init="",
                         classnames=["class 0", "class 1", "dog", "sun flower", "y"], batch=2, kind="noise"),
}


def run_variant_case(name: str, spec: dict, out_dir: str) -> None:
    """Unmodified reference trainers/{umudpt,uumudpt}.py CustomCLIP; every trainable tensor = syn.param_by_name."""
    clip_pkg, clip_model_mod, _ = ref_shims.import_reference()
    ref_mod = ref_shims.import_reference_variant(spec["trainer"])
    arch = syn.ARCHS[spec["arch"]]
    cfg = ref_shims.make_cfg(n_ctx=spec["n_ctx"], depth=spec["depth"], ctx_init=spec["ctx_init"], size=arch.image_resolution,
                             name=spec["trainer"])
    t0 = time.time()
    clip_model = clip_model_mod.CLIP(*arch.astuple(), cfg).float()
    clip_model.load_state_dict(syn.synthetic_clip_state_dict(arch, seed=0), strict=False)
    model = ref_mod.CustomCLIP(cfg, spec["classnames"], clip_model)
    keep_vis = spec["trainer"] == "UUMuDPT"
    for n, p in model.named_parameters():   # trainers/umudpt.py:250-253, uumudpt.py:252-261
        if "prompt_learner" not in n:
            p.requires_grad_(keep_vis and "visual_ctx" in n)
    with torch.no_grad():
        for n, p in model.named_parameters():
            if p.requires_grad and not (n.endswith("prompt_learner.ctx") and spec["ctx_init"]):
                p.copy_(syn.param_by_name(n, p.shape, seed=0))
    tokenized = model.tokenized_prompts.clone()
    ctx_tokens = clip_pkg.tokenize(spec["ctx_init"].replace("_", " "))[0] if spec["ctx_init"] else None
    image = syn.synthetic_images(spec["batch"], arch.image_resolution, seed=1, kind=spec["kind"])
    labels = syn.synthetic_labels(spec["batch"], len(spec["classnames"]), seed=1)
    model.zero_grad()
    logits = model(image)
    loss = F.cross_entropy(logits, labels)
    loss.backward()
    out = {
        "trainer": np.array(spec["trainer"]), "arch": np.array(spec["arch"]), "n_ctx": np.array(spec["n_ctx"]),
        "depth": np.array(spec["depth"]), "batch": np.array(spec["batch"]), "kind": np.array(spec["kind"]),
        "classnames": np.array(spec["classnames"]), "ctx_init": np.array(spec["ctx_init"]),
        "ctx_init_tokens": (ctx_tokens.numpy() if ctx_tokens is not None else np.zeros(0, np.int32)),
        "tokenized_prompts": tokenized.numpy().astype(np.int32), "labels": labels.numpy(),
        "logits": logits.detach().numpy(), "loss": loss.detach().numpy(),
        "state_keys": np.array(sorted(model.state_dict().keys())),
    }
    for n, p in model.named_parameters():
        if p.requires_grad:
            out["grad/" + n] = p.grad.numpy()
    path = os.path.join(out_dir, name + ".npz")
    gu.save(path, out)
    print(f"{name}: loss={float(loss.detach()):.6f} logits{tuple(logits.shape)} trainable={sum(1 for k in out if k.startswith('grad/'))} "
          f"-> {path} ({os.path.getsize(path)/1e6:.2f} MB, {time.time()-t0:.1f}s)")


def main():
    out_dir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    which = sys.argv[1:] or (list(CASES) + list(COCOOP_CASES) + list(VARIANT_CASES))
    for name in which:
        if name in VARIANT_CASES:
            run_variant_case(name, VARIANT_CASES[name], out_dir)
        elif name in COCOOP_CASES:
            run_cocoop_case(name, COCOOP_CASES[name], out_dir)
        else:
            run_case(name, CASES[name], out_dir)


if __name__ == "__main__":
    main()

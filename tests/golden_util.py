"""Load a golden fixture (made from the reference by oracle/make_golden.py) and rebuild the
exact synthetic state dict it was produced with."""
import os

import numpy as np
import torch

from mudpt_b200 import synthetic as syn

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TINY = ["tiny_a", "tiny_b", "tiny_c", "tiny_d"]
LOWRANK = "lowrank/"  # lowrank/<key>/a and lowrank/<key>/b stand for the array <key> = a @ b

_cache = {}


def save(path, arrays):
    """np.savez_compressed, except that a large 2-D gradient of low numerical rank r (the weight gradient of a
    projection applied to a few prompt rows) is stored as two rank-r factors when they take less than half its
    space, which keeps the ViT-B/16 fixture small.  Their product equals the gradient to fp32 rounding."""
    out = {}
    for k, v in arrays.items():
        if k.startswith("grad/") and v.ndim == 2 and v.dtype == np.float32 and v.size >= 4096:
            u, s, vt = np.linalg.svd(v.astype(np.float64), full_matrices=False)
            r = int((s > 1e-6 * s[0]).sum())
            if 2 * r * sum(v.shape) < v.size:
                a, b = (u[:, :r] * s[:r]).astype(np.float32), vt[:r].astype(np.float32)
                if np.abs(a.astype(np.float64) @ b - v).max() <= 1e-6 * np.abs(v).max():
                    out[LOWRANK + k + "/a"], out[LOWRANK + k + "/b"] = a, b
                    continue
        out[k] = v
    np.savez_compressed(path, **out)


def _read(name):
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False)
    g = {k: z[k] for k in z.files if not k.startswith(LOWRANK)}
    for k in z.files:
        if k.startswith(LOWRANK) and k.endswith("/a"):
            g[k[len(LOWRANK):-2]] = (z[k].astype(np.float64) @ z[k[:-1] + "b"]).astype(np.float32)
    return g


def load(name):
    if name in _cache:
        return _cache[name]
    g = _read(name)
    arch = syn.ARCHS[str(g["arch"])]
    n_ctx, depth, batch = int(g["n_ctx"]), int(g["depth"]), int(g["batch"])
    tok = torch.from_numpy(g["tokenized_prompts"])
    ctx_tokens = torch.from_numpy(g["ctx_init_tokens"]) if bool(g["has_ctx_init"]) else None
    sd = syn.assemble_state_dict(arch, tok, n_ctx, depth, ctx_tokens, seed=0)
    image = syn.synthetic_images(batch, arch.image_resolution, seed=1, kind=str(g["kind"]))
    labels = torch.from_numpy(g["labels"])
    case = dict(arch=arch, n_ctx=n_ctx, depth=depth, batch=batch, sd=sd, tokenized=tok, image=image,
                labels=labels, golden=g, classnames=[str(c) for c in g["classnames"]])
    _cache[name] = case
    return case


make_cfg = syn.make_cfg  # the yacs subset the hot path reads lives with the product (bench.py uses it too)


def build_model(case, device="cuda"):
    """mudpt_b200 CustomCLIP carrying exactly the golden case's weights (token ids from the fixture)."""
    from mudpt_b200 import clip
    from mudpt_b200.trainers.mudpt import CustomCLIP
    g = case["golden"]
    arch = case["arch"]
    ctx_init = "a photo of a" if bool(g["has_ctx_init"]) else ""
    cfg = make_cfg(case["n_ctx"], case["depth"], ctx_init, arch.image_resolution)
    prefix = " ".join(ctx_init.split()[:case["n_ctx"]]) if ctx_init else " ".join(["X"] * case["n_ctx"])
    table = {prefix + " " + n.replace("_", " ") + ".": case["tokenized"][i:i + 1] for i, n in enumerate(case["classnames"])}
    if ctx_init:
        table[ctx_init] = torch.from_numpy(g["ctx_init_tokens"]).view(1, -1)
    clip_model = clip.CLIP(*arch.astuple(), cfg).float()
    model = CustomCLIP(cfg, case["classnames"], clip_model, tokenizer=lambda s: table[s])
    missing = model.load_state_dict(case["sd"], strict=True)
    for n, p in model.named_parameters():
        if "prompt_learner" not in n:
            p.requires_grad_("visual_ctx" in n)
    return model.to(device), cfg


COCOOP = ["cocoop_tiny_a", "cocoop_tiny_b"]


def load_cocoop(name):
    """CoCoOp fixture (BASELINE config 4) made from the reference's trainers/cocoop.py."""
    if name in _cache:
        return _cache[name]
    g = _read(name)
    arch = syn.ARCHS[str(g["arch"])]
    n_ctx, batch = int(g["n_ctx"]), int(g["batch"])
    tok = torch.from_numpy(g["tokenized_prompts"])
    ctx_tokens = torch.from_numpy(g["ctx_init_tokens"]) if bool(g["has_ctx_init"]) else None
    sd = syn.assemble_cocoop_state_dict(arch, tok, n_ctx, ctx_tokens, seed=0)
    image = syn.synthetic_images(batch, arch.image_resolution, seed=1, kind=str(g["kind"]))
    case = dict(arch=arch, n_ctx=n_ctx, batch=batch, sd=sd, tokenized=tok, image=image, labels=torch.from_numpy(g["labels"]),
                golden=g, classnames=[str(c) for c in g["classnames"]], ctx_init=str(g["ctx_init"]))
    _cache[name] = case
    return case


def make_cocoop_cfg(n_ctx, ctx_init, size, arch_name="ViT-B/16"):
    cfg = make_cfg(n_ctx, 1, ctx_init, size, arch_name)
    cfg.TRAINER["NAME"] = "CoCoOp"
    cfg.TRAINER["COCOOP"] = type(cfg)(N_CTX=n_ctx, CTX_INIT=ctx_init, PREC="fp32")
    return cfg


def build_cocoop_model(case, device="cuda"):
    """mudpt_b200 CoCoOp CustomCLIP carrying exactly the golden case's weights (token ids from the fixture)."""
    from mudpt_b200 import clip
    from mudpt_b200.trainers.cocoop import CustomCLIP
    g, arch = case["golden"], case["arch"]
    ctx_init = case["ctx_init"]
    cfg = make_cocoop_cfg(case["n_ctx"], ctx_init, arch.image_resolution)
    prefix = ctx_init if ctx_init else " ".join(["X"] * case["n_ctx"])
    table = {prefix + " " + n.replace("_", " ") + ".": case["tokenized"][i:i + 1] for i, n in enumerate(case["classnames"])}
    if ctx_init:
        table[ctx_init] = torch.from_numpy(g["ctx_init_tokens"]).view(1, -1)
    clip_model = clip.CLIP(*arch.astuple(), None).float()
    model = CustomCLIP(cfg, case["classnames"], clip_model, tokenizer=lambda s: table[s])
    model.load_state_dict(case["sd"], strict=True)
    for n, p in model.named_parameters():
        if "prompt_learner" not in n:
            p.requires_grad_(False)
    return model.to(device), cfg


VARIANTS = ["umudpt_tiny", "uumudpt_tiny"]


def load_variant(name):
    """UMuDPT / UUMuDPT fixture (SURVEY 8f N4) made from the reference's trainers/{umudpt,uumudpt}.py."""
    if name in _cache:
        return _cache[name]
    g = _read(name)
    arch = syn.ARCHS[str(g["arch"])]
    case = dict(trainer=str(g["trainer"]), arch=arch, n_ctx=int(g["n_ctx"]), depth=int(g["depth"]), batch=int(g["batch"]),
                tokenized=torch.from_numpy(g["tokenized_prompts"]), labels=torch.from_numpy(g["labels"]),
                image=syn.synthetic_images(int(g["batch"]), arch.image_resolution, seed=1, kind=str(g["kind"])),
                golden=g, classnames=[str(c) for c in g["classnames"]], ctx_init=str(g["ctx_init"]))
    _cache[name] = case
    return case


def build_variant_model(case, device="cuda"):
    """mudpt_b200 UMuDPT / UUMuDPT CustomCLIP with the fixture's weights: synthetic CLIP state dict, every trainable
    tensor = syn.param_by_name (ctx from the token embedding when CTX_INIT is given), token ids from the fixture."""
    import importlib
    from mudpt_b200 import clip
    g, arch, name = case["golden"], case["arch"], case["trainer"]
    mod = importlib.import_module("mudpt_b200.trainers." + name.lower())
    ctx_init = case["ctx_init"]
    cfg = make_cfg(case["n_ctx"], case["depth"], ctx_init, arch.image_resolution)
    cfg.TRAINER["NAME"] = name
    cfg.TRAINER[name.upper()] = type(cfg)(N_CTX=case["n_ctx"], CTX_INIT=ctx_init, DEEP_PROMPT_DEPTH=case["depth"], PREC="fp32")
    prefix = " ".join(ctx_init.split()[:case["n_ctx"]]) if ctx_init else " ".join(["X"] * case["n_ctx"])
    table = {prefix + " " + n.replace("_", " ") + ".": case["tokenized"][i:i + 1] for i, n in enumerate(case["classnames"])}
    if ctx_init:
        table[ctx_init] = torch.from_numpy(g["ctx_init_tokens"]).view(1, -1)
    clip_model = clip.CLIP(*arch.astuple(), cfg).float()
    clip_model.load_state_dict(syn.synthetic_clip_state_dict(arch, 0), strict=False)
    model = mod.CustomCLIP(cfg, case["classnames"], clip_model, tokenizer=lambda s: table[s])
    keep_vis = name == "UUMuDPT"
    for n, p in model.named_parameters():
        if "prompt_learner" not in n:
            p.requires_grad_(keep_vis and "visual_ctx" in n)
    with torch.no_grad():
        for n, p in model.named_parameters():
            if p.requires_grad and not (n.endswith("prompt_learner.ctx") and ctx_init):
                p.copy_(syn.param_by_name(n, p.shape, seed=0))
    return model.to(device), cfg

"""Tower parity stage by stage, at the shapes the towers run (`-m gpu`).

One training forward of a full-depth tower on the synthetic weights; then every stage of every block is checked against
fp64 computed from the tower's own saved operands (Engine.debug_buffer), with the per-block unit-test bounds
(tests/tower_stages.py has the table).  The whole-model checks (feature cosine, logit and gradient error after 12 layers)
dilute a fault of one layer, one stage or one 128-row band through the rest of the tower; these do not.  Covered here,
at the shapes where they run: the fused LayerNorm chain (statistics from the previous block's residual epilogue, under
stream-K), the deep-prompt splice inside that epilogue, the pruned last block (gathered CLS / EOT rows), the ragged text
tower (packed rows, per-class lse), the patch-embedding stem (EPI_PATCH) and the tcgen05 attention kernels over the
workspace qkv.  Every layer of every configuration is checked, the 77,000-row text tower included.

The backward keeps no per-layer gradients; it is checked through 3-layer towers at the real widths and row counts
(test_backward_depth3): block-0 work skipping, the pruned last block and the scatter of its rows, the ragged LayerNorm
backward window, the bf16 gradient stream, the fused LayerNorm dgrad (EPI_LN_BWD), the image gradient through the stem.

Each configuration prints its worst block ratio (error / bound) per stage and the (layer, block) where it occurs."""
import dataclasses

import pytest
import torch
import torch.nn.functional as F

from tests import tower_stages as ts
from tests.test_gpu_parity import F32_REL

pytestmark = pytest.mark.gpu

VISION, TEXT = 0, 1

# name -> configuration; ViT-B/16, n_ctx 2, prompt depth 9 unless noted
FORWARD = {
    "vitb16_b32": dict(tower="vision", B=32),                       # 6368 rows, stand-alone LayerNorm, pair tiles
    "vitb16_b165": dict(tower="vision", B=165),                     # 32,835 rows: fused LayerNorm by the row threshold
    "vitb16_b32_ln_fused": dict(tower="vision", B=32, ln_fused=1),
    "vitb16_b32_prune0": dict(tower="vision", B=32, prune=0),
    "vitb32_b32": dict(tower="vision", arch="ViT-B/32", B=32),      # 52 tokens, K = 3072 stem
    "vitl14_b8": dict(tower="vision", arch="ViT-L/14", B=8, depth=12),  # 259 tokens, d = 1024, Kp = 592
    "text_125x77": dict(tower="text", C=125, mode=False),           # 9625 rows, stand-alone LayerNorm
    "text_1000x77": dict(tower="text", C=1000, mode=False),         # 77,000 rows, fused chain
    "text_1000_eot": dict(tower="text", C=1000, mode=True),
    "text_ragged_long": dict(tower="text", C=250, mode="per_class", names="long"),
    "text_plain": dict(tower="text", C=125, mode=False, n_ctx=0, depth=1),
}


@pytest.fixture(scope="module")
def engines():
    """(Engine, state dict, arch) per (arch, n_ctx, depth), built once for the module."""
    from mudpt_b200 import synthetic as syn
    from mudpt_b200.engine import Engine
    cache = {}

    def get(arch_name, n_ctx, depth, layers=None):
        key = (arch_name, n_ctx, depth, layers)
        if key not in cache:
            arch = syn.ARCHS[arch_name]
            if layers is not None:
                arch = dataclasses.replace(arch, vision_layers=layers, transformer_layers=layers)
            sd = syn.synthetic_clip_state_dict(arch, 0)
            eng = Engine(dataclasses.asdict(arch), n_ctx, depth, torch.device("cuda"))
            eng.load_clip_weights(sd)
            cache[key] = (eng, sd, arch)
        return cache[key]
    yield get
    cache.clear()


def _opt(eng, name, value):
    from mudpt_b200 import _lib
    _lib.check(eng.lib.mudpt_set_option(eng.h, name.encode(), value), eng.h)


def _ops(eng, tower, d):
    """ops(name, layer) of tower_stages: the saved buffer as [rows, width] (lse flat), cached for the layer pair in use"""
    width = {"x_in": d, "x_mid": d, "qkv": 3 * d, "o": d, "h": 4 * d}
    cache = {}

    def ops(name, i):
        if (name, i) not in cache:
            if len(cache) > 8:
                cache.clear()
            dt = torch.float32 if name in ("x_in", "x_mid", "lse") else torch.bfloat16
            t = eng.debug_buffer(tower, name, i, dt)
            cache[name, i] = t if name == "lse" else t.view(-1, width[name])
        return cache[name, i]
    return ops


def _weights(sd, prefix, dev):
    return lambda i: {k: sd[f"{prefix}{i}.{k}"].to(dev) for k in ts.BLOCK_KEYS}


def _vision(engines, cfg):
    from mudpt_b200 import synthetic as syn
    n_ctx, depth = cfg.get("n_ctx", 2), cfg.get("depth", 9)
    eng, sd, arch = engines(cfg.get("arch", "ViT-B/16"), n_ctx, depth)
    dev, B, d, p = torch.device("cuda"), cfg["B"], arch.vision_width, arch.vision_patch_size
    _opt(eng, "prune", cfg.get("prune", 1))
    _opt(eng, "ln_fused", cfg.get("ln_fused", -1))
    g = torch.Generator().manual_seed(B)
    prompts = torch.randn(depth, n_ctx, d, generator=g).to(dev)  # ln_pre-scale rows, like the prompt stack's
    img = syn.synthetic_images(B, arch.image_resolution, seed=B).to(dev)
    f = eng.vision_forward(img, prompts)
    torch.cuda.synchronize()
    npatch = (arch.image_resolution // p) ** 2
    L = 1 + npatch + n_ctx
    rows = B * L
    geo = ts.Geometry(lengths=[L] * B, H=d // 64, causal=False, row0=1 + npatch, n_ctx=n_ctx,
                      spliced=list(range(depth)) if n_ctx else [], sel=[b * L for b in range(B)])
    ops = _ops(eng, VISION, d)
    rep = ts.Report()
    # stem: ln_pre(conv1 as a GEMM of the bf16 patches and weight + pos; CLS + pos), every row but the prompt rows
    V = "visual."
    pat = F.unfold(img, kernel_size=p, stride=p).transpose(1, 2).bfloat16().double()
    W = sd[V + "conv1.weight"].to(dev).reshape(d, -1).bfloat16().double()
    pos = sd[V + "positional_embedding"].to(dev).double()
    x0 = torch.empty(B, L, d, device=dev, dtype=torch.float64)
    x0[:, 0] = sd[V + "class_embedding"].to(dev).double() + pos[0]
    x0[:, 1:1 + npatch] = pat @ W.t() + pos[1:]
    x0 = F.layer_norm(x0[:, :1 + npatch], (d,), sd[V + "ln_pre.weight"].to(dev).double(), sd[V + "ln_pre.bias"].to(dev).double(), ts.LN_EPS)
    got = ops("x_in", 0).view(B, L, d)[:, :1 + npatch]
    rep.add(0, "stem", *ts.per_row(got.reshape(-1, d), x0.reshape(-1, d), F32_REL, lambda i: (i // (1 + npatch), i % (1 + npatch))))
    fused = cfg.get("ln_fused", -1) == 1 or rows >= 32768
    return ts.check_tower(ops, _weights(sd, V + "transformer.resblocks.", dev), arch.vision_layers, geo, prompts, fused,
                          bool(cfg.get("prune", 1)), f, sd[V + "ln_post.weight"].to(dev), sd[V + "ln_post.bias"].to(dev),
                          sd[V + "proj"].to(dev), rep=rep)


def _text(engines, cfg):
    from mudpt_b200 import synthetic as syn
    from mudpt_b200.engine import packed_offsets, text_lengths
    n_ctx, depth = cfg.get("n_ctx", 2), cfg.get("depth", 9)
    eng, sd, arch = engines("ViT-B/16", n_ctx, depth)
    dev, C, d, mode = torch.device("cuda"), cfg["C"], arch.transformer_width, cfg["mode"]
    _opt(eng, "prune", cfg.get("prune", 1))
    _opt(eng, "ln_fused", cfg.get("ln_fused", -1))
    names = syn.synthetic_classnames(C, cfg.get("names", "short"))
    tok = syn.synthetic_tokenize([" ".join(["X"] * n_ctx + [n]) + "." for n in names])
    eot = tok.argmax(-1)
    g = torch.Generator().manual_seed(C)
    emb = torch.randn(C, arch.context_length, d, generator=g) * 0.02
    seq_len, lengths = text_lengths(eot, mode, arch.context_length, 1 + n_ctx)
    eng.text_set_classes(emb, eot, seq_len, lengths)
    lengths = lengths or [seq_len] * C
    prompts = (torch.randn(depth, n_ctx, d, generator=g) * 0.02).to(dev)
    f = eng.text_forward(prompts, True)
    torch.cuda.synchronize()
    off = packed_offsets(lengths)
    geo = ts.Geometry(lengths=lengths, H=arch.transformer_heads, causal=True, row0=1, n_ctx=n_ctx,
                      spliced=list(range(depth)) if n_ctx else [], sel=[off[c] + int(eot[c]) for c in range(C)])
    ops = _ops(eng, TEXT, d)
    rep = ts.Report()
    # stem: token embedding + positional embedding on every row but the prompt rows
    cls = torch.repeat_interleave(torch.arange(C), torch.tensor(lengths))
    tpos = torch.cat([torch.arange(n) for n in lengths])
    ref = (emb[cls, tpos].double() + sd["positional_embedding"][tpos].double()).to(dev)
    keep = torch.ones(off[-1], dtype=torch.bool, device=dev)
    if n_ctx:
        keep[geo.prompt_rows(dev).flatten()] = False
    rows = keep.nonzero().flatten()
    rep.add(0, "stem", *ts.per_row(ops("x_in", 0)[rows], ref[rows], F32_REL, lambda i: (int(rows[i]),)))
    fused = mode != "per_class" and (cfg.get("ln_fused", -1) == 1 or off[-1] >= 32768)
    return ts.check_tower(ops, _weights(sd, "transformer.resblocks.", dev), arch.transformer_layers, geo, prompts, fused,
                          bool(cfg.get("prune", 1)), f, sd["ln_final.weight"].to(dev), sd["ln_final.bias"].to(dev),
                          sd["text_projection"].to(dev), rep=rep)


@pytest.mark.parametrize("name", list(FORWARD))
def test_forward_stages(engines, name):
    """Teacher-forced forward: stem, splice, LN1 + in-proj, attention (o and lse), out-proj + residual, LN2 + c_fc,
    c_proj + residual of every block, and the pruned last block / the feature head, each against fp64 from the tower's
    own operands at the bound of the kernel that computed it."""
    cfg = FORWARD[name]
    rep = (_vision if cfg["tower"] == "vision" else _text)(engines, cfg)
    print()
    print(rep.table(name), flush=True)
    assert rep.failures() == [], (name, rep.failures()[:8])


# ------------------------------------------------------------------------------------------------ backward
# 3-layer towers at the real widths and row counts, prompt depth 3: block 0 (work skipping onto the prompt rows), a middle
# block (full dgrad) and the last block (pruned or not).  Every value of prune, grad_stream_bf16 and ln_fused on each
# tower, ln_bwd_fused = 1 once (options not named take their defaults: ln_fused by row count, ln_bwd_fused 0,
# grad_stream_bf16 1).
BACKWARD = {
    "vitb16_b32": dict(tower="vision", B=32),                                     # stand-alone LayerNorm, block-0 skipping
    "vitb16_b32_images": dict(tower="vision", B=32, prune=0, images=True),         # d_images (fp32 stream: need_dx0)
    "vitb16_b165": dict(tower="vision", B=165, ln_bwd_fused=1),                   # fused chain, LayerNorm dgrad in the GEMMs
    "vitl14_b4": dict(tower="vision", arch="ViT-L/14", B=4, prune=0, gs=0, ln_fused=1),
    "text_125x77": dict(tower="text", C=125, mode=False),
    "text_1000x77": dict(tower="text", C=1000, mode=False, prune=0, gs=0),         # 77,000 rows, fused chain
    "text_125x77_dx0": dict(tower="text", C=125, mode=False, ln_fused=1, dx0=True),
    "text_ragged_long": dict(tower="text", C=250, mode="per_class", names="long"),  # packed LayerNorm backward window
}
BWD_LAYERS, BWD_DEPTH = 3, 3


def _set_options(eng, cfg):
    for k, v in (("prune", cfg.get("prune", 1)), ("ln_fused", cfg.get("ln_fused", -1)),
                 ("ln_bwd_fused", cfg.get("ln_bwd_fused", 0)), ("grad_stream_bf16", cfg.get("gs", 1))):
        _opt(eng, k, v)


def _ln_x16(cfg, fused):
    """The LayerNorm backwards that read the bf16 row after a fused forward: all of them, except the pruned last block's
    LN2 when the LayerNorm backward runs stand-alone (it reads the gathered fp32 rows)"""
    if not fused:
        return frozenset()
    keep_fp32 = {(BWD_LAYERS - 1, 2)} if cfg.get("prune", 1) and not cfg.get("ln_bwd_fused", 0) else set()
    return frozenset((i, k) for i in range(BWD_LAYERS) for k in (1, 2)) - keep_fp32


def _leaf(t):
    return t.detach().double().clone().requires_grad_(True)


def _backward_vision(engines, cfg):
    from mudpt_b200 import synthetic as syn
    eng, sd, arch = engines(cfg.get("arch", "ViT-B/16"), 2, BWD_DEPTH, BWD_LAYERS)
    _set_options(eng, cfg)
    dev, B, d, p = torch.device("cuda"), cfg["B"], arch.vision_width, arch.vision_patch_size
    n_ctx, R = 2, arch.image_resolution
    g = torch.Generator().manual_seed(B + 1)
    prompts = torch.randn(BWD_DEPTH, n_ctx, d, generator=g).to(dev)
    img = syn.synthetic_images(B, R, seed=B).to(dev)
    eng.vision_forward(img, prompts)
    d_f = torch.randn(B, arch.embed_dim, generator=g).to(dev)
    x0 = eng.debug_buffer(VISION, "x_in", 0, torch.float32).view(-1, d)
    if cfg.get("images"):
        dP, d_img = eng.vision_backward_images(d_f)
    else:
        dP = eng.vision_backward(d_f)
    torch.cuda.synchronize()
    npatch = (R // p) ** 2
    L = 1 + npatch + n_ctx
    geo = ts.Geometry(lengths=[L] * B, H=d // 64, causal=False, row0=1 + npatch, n_ctx=n_ctx, spliced=list(range(BWD_DEPTH)),
                      sel=[b * L for b in range(B)])
    V = "visual."
    fused = cfg.get("ln_fused", -1) == 1 or B * L >= 32768
    need_dx0 = bool(cfg.get("images"))
    gs = bool(cfg.get("gs", 1)) and not (fused and cfg.get("ln_bwd_fused", 0)) and not need_dx0
    grads = {}
    for emulate in (False, True):
        dt = torch.float32 if emulate else torch.float64
        P = _leaf(prompts).to(dt).detach().requires_grad_(True)
        if need_dx0:
            # the stem from the (bf16-rounded) pixels: ln_pre(conv1 patches + pos; CLS + pos); its input gradient is bf16
            im = img.bfloat16().to(dt).requires_grad_(True)
            pat = F.unfold(im, kernel_size=p, stride=p).transpose(1, 2)
            Wc = sd[V + "conv1.weight"].to(dev).reshape(d, -1)
            pos = sd[V + "positional_embedding"].to(dev).to(dt)
            cls = (sd[V + "class_embedding"].to(dev).to(dt) + pos[0]).expand(B, 1, d)
            xp = pat @ (Wc.bfloat16() if emulate else Wc).to(dt).t() + pos[1:]
            xs = torch.cat([cls, xp, torch.zeros(B, n_ctx, d, device=dev, dtype=dt)], 1).reshape(-1, d)
            if emulate:
                xs = ts._Round.apply(xs, False, True)
            xin = F.layer_norm(xs, (d,), sd[V + "ln_pre.weight"].to(dev).to(dt), sd[V + "ln_pre.bias"].to(dev).to(dt), ts.LN_EPS)
        else:
            im, xin = None, x0.to(dt)
        ts.tower_grads(xin, P, _weights(sd, V + "transformer.resblocks.", dev), BWD_LAYERS, geo, sd[V + "ln_post.weight"].to(dev),
                       sd[V + "ln_post.bias"].to(dev), sd[V + "proj"].to(dev), d_f, emulate, gs and emulate, _ln_x16(cfg, fused))
        grads[emulate] = (P.grad, im.grad if im is not None else None)
    rep = ts.Report()
    nrow = BWD_DEPTH * n_ctx
    r, blk = ts.grad_blocks(dP.view(nrow, d), grads[False][0].view(nrow, d), grads[True][0].view(nrow, d), (nrow,),
                            lambda i: (i // n_ctx, i % n_ctx))
    rep.add(blk[0], "d_prompts", r, blk)
    if need_dx0:
        gh = R // p

        def bands(t):  # [B, 3, R, R] -> one block per (image, patch-row band)
            return t.reshape(B, 3, gh, p, R).permute(0, 2, 1, 3, 4).reshape(B * gh, -1)
        r, blk = ts.grad_blocks(bands(d_img), bands(grads[False][1]), bands(grads[True][1]), (B * gh,), lambda i: (i // gh, i % gh))
        rep.add(0, "d_images", r, blk)
    return rep


def _backward_text(engines, cfg):
    from mudpt_b200 import synthetic as syn
    from mudpt_b200.engine import packed_offsets, text_lengths
    eng, sd, arch = engines("ViT-B/16", 2, BWD_DEPTH, BWD_LAYERS)
    _set_options(eng, cfg)
    dev, C, d, mode, n_ctx = torch.device("cuda"), cfg["C"], arch.transformer_width, cfg["mode"], 2
    names = syn.synthetic_classnames(C, cfg.get("names", "short"))
    eot = syn.synthetic_tokenize([" ".join(["X"] * n_ctx + [n]) + "." for n in names]).argmax(-1)
    g = torch.Generator().manual_seed(C + 1)
    emb = torch.randn(C, arch.context_length, d, generator=g) * 0.02
    seq_len, lengths = text_lengths(eot, mode, arch.context_length, 1 + n_ctx)
    eng.text_set_classes(emb, eot, seq_len, lengths)
    lengths = lengths or [seq_len] * C
    prompts = (torch.randn(BWD_DEPTH, n_ctx, d, generator=g) * 0.02).to(dev)
    eng.text_forward(prompts, True)
    d_f = torch.randn(C, arch.embed_dim, generator=g).to(dev)
    x0 = eng.debug_buffer(TEXT, "x_in", 0, torch.float32).view(-1, d)
    need_dx0 = bool(cfg.get("dx0"))
    dP, dx0 = eng.text_backward(d_f, need_dx0)
    torch.cuda.synchronize()
    off = packed_offsets(lengths)
    geo = ts.Geometry(lengths=lengths, H=arch.transformer_heads, causal=True, row0=1, n_ctx=n_ctx, spliced=list(range(BWD_DEPTH)),
                      sel=[off[c] + int(eot[c]) for c in range(C)])
    fused = mode != "per_class" and (cfg.get("ln_fused", -1) == 1 or off[-1] >= 32768)
    gs = bool(cfg.get("gs", 1)) and not (fused and cfg.get("ln_bwd_fused", 0)) and not need_dx0
    grads = {}
    for emulate in (False, True):
        dt = torch.float32 if emulate else torch.float64
        P = _leaf(prompts).to(dt).detach().requires_grad_(True)
        x = x0.to(dt).requires_grad_(True)
        ts.tower_grads(x, P, _weights(sd, "transformer.resblocks.", dev), BWD_LAYERS, geo, sd["ln_final.weight"].to(dev),
                       sd["ln_final.bias"].to(dev), sd["text_projection"].to(dev), d_f, emulate, gs and emulate, _ln_x16(cfg, fused))
        grads[emulate] = (P.grad, x.grad)
    rep = ts.Report()
    nrow = BWD_DEPTH * n_ctx
    r, blk = ts.grad_blocks(dP.view(nrow, d), grads[False][0].view(nrow, d), grads[True][0].view(nrow, d), (nrow,),
                            lambda i: (i // n_ctx, i % n_ctx))
    rep.add(blk[0], "d_prompts", r, blk)
    if need_dx0:
        # the layer-0 prompt rows' gradient went to d_prompts[0]: every other row of the (padded) tower input
        keep = torch.ones(off[-1], dtype=torch.bool, device=dev)
        keep[geo.prompt_rows(dev).flatten()] = False
        rows = keep.nonzero().flatten()
        got = dx0.reshape(-1, d)[rows]
        r, blk = ts.grad_blocks(got, grads[False][1][rows], grads[True][1][rows], (rows.numel(),), lambda i: (int(rows[i]),))
        rep.add(0, "d_x0", r, blk)
    return rep


@pytest.mark.parametrize("name", list(BACKWARD))
def test_backward_depth3(engines, name):
    """Prompt gradients per (layer, token) row, the dense input gradient per row (text, want_dx0) and the image gradient
    per (image, patch-row band) of a 3-layer tower against fp64 autograd from the tower's own x_in[0] (vision images: from
    the pixels through the stem) and the same d_f, each block bounded by max(BF16_REL, 1.6 x the error of the fp32
    emulation with the native roundings on that block) (tests/tower_stages.py, tower_grads)."""
    cfg = BACKWARD[name]
    rep = (_backward_vision if cfg["tower"] == "vision" else _backward_text)(engines, cfg)
    print()
    print(rep.table(name + " (backward)"), flush=True)
    assert rep.failures() == [], (name, rep.failures())

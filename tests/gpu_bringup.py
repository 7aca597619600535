"""GPU bring-up / diagnostics driver (run on the B200 box through gpurun).

    python tests/gpu_bringup.py [group ...]      # default: all groups

Every group runs in its own subprocess under a timeout, so a trapping kernel cannot poison
the other groups (a CUDA fault is sticky for its process).  Results go to stdout and to
gpurun_out/bringup.json.  This is test infrastructure: it compares the native kernels with
plain torch fp32 math on the same device and with the golden fixtures made from the reference.
"""
from __future__ import annotations

import json
import math
import os
import subprocess
import sys
import time
import traceback

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

GROUPS = ["gemm", "gemm_fused", "rowops", "attention", "head", "model_tiny", "model_vitb16"]


# A kernel bug on one path (an M tail, the last partial wave, one stream-K hand-over, one (sequence, head) problem) touches
# one tile or row band and is diluted by everything that is correct in a whole-tensor norm.  Bounds are therefore applied
# per block.  A block whose reference is near zero (e.g. the last keys' dk under a causal mask) carries the rounding of
# the whole computation, not its own scale: its denominator is floored at BLK_FLOOR x (RMS of the reference) x sqrt(n).
# The floor follows the whole tensor: where block scales differ by design (the head's per-class d f_txt: a few label
# classes carry most of the gradient), compare the groups as separate tensors so each is floored at its own scale.
BLK_FLOOR = 0.25
GEMM_TILE = (128, 128)
# elementwise bound of a bf16-operand GEMM against the fp64 product of the same operands (see _gemm_elementwise):
# |out - ref| <= BF16_OUT_ROUND |ref| (bf16 outputs) + ELEM_C[type] 2^-24 (sqrt(K) (|A| |B|^T) + |bias| + |resid|)
BF16_OUT_ROUND = 2.0 ** -8
ELEM_C = {"bf16": 4.0, "f32": 4.0}
GUARD = 8  # rows after an output that a kernel must leave alone


def _metrics(a, b, tile=None, grid=None):
    """Whole-tensor parity of `a` against the reference `b` plus, with a block layout, the worst block.

    tile=(tm, tn): a and b are 2-D; blocks are tm x tn tiles (the shape is padded to whole tiles), blk_worst = the
    first (row, column) of the worst tile.  grid=(g0, g1, ...): a and b are viewed as [g0 * g1 * ..., -1], one block
    per row of that view, blk_worst = the grid index of the worst block."""
    import torch
    af = a.double().flatten()
    bf = b.double().flatten()
    d = (af - bf)
    m = {"cos": float((af @ bf) / (af.norm() * bf.norm() + 1e-300)), "rel": float(d.norm() / (bf.norm() + 1e-300)),
         "max_abs": float(d.abs().max()), "ref_max": float(bf.abs().max()), "nan": bool(torch.isnan(af).any())}
    if tile is None and grid is None:
        return m
    blk = _block_rel(a, b, tile, grid)
    i = int(blk.argmax())
    m["blk_rel"] = float(blk[i])
    if tile is not None:
        cols = -(-b.shape[1] // tile[1])
        m["blk_worst"] = [(i // cols) * tile[0], (i % cols) * tile[1]]
    else:
        m["blk_worst"] = [int(v) for v in torch.unravel_index(torch.tensor(i), grid)]
    return m


def _block_rel(a, b, tile=None, grid=None):
    """Relative L2 error of every block (flat, in block order) of `a` against `b`; layouts as in _metrics."""
    import torch
    bf = b.double().flatten()
    if tile is not None:
        import torch.nn.functional as F
        tm, tn = tile
        M, N = b.shape
        pad = (0, -N % tn, 0, -M % tm)

        def per_block(x):
            x = F.pad(x, pad)
            return x.view(x.shape[0] // tm, tm, x.shape[1] // tn, tn).sum((1, 3)).flatten()
        dd, a2 = (a.double() - b.double()), b.double()
        e2, r2, n = per_block(dd * dd), per_block(a2 * a2), per_block(torch.ones_like(a2))
    else:
        nb = math.prod(grid)
        dd, a2 = (a.double() - b.double()).reshape(nb, -1), b.double().reshape(nb, -1)
        e2, r2 = (dd * dd).sum(1), (a2 * a2).sum(1)
        n = torch.full_like(e2, a2.shape[1])
    rms2 = float((bf * bf).mean()) if bf.numel() else 0.0
    den = torch.maximum(r2, (BLK_FLOOR ** 2) * rms2 * n).clamp_min(1e-300)
    blk = (e2 / den).sqrt()
    return torch.where(torch.isnan(blk), torch.full_like(blk, float("inf")), blk)  # an unwritten (NaN) element fails its block


def _gemm_elementwise(out, ref, A, B, kind, bias=None, resid=None):
    """max over the output of |out - ref| / bound for C = A B^T (+ bias + resid), `ref` computed in fp64 from the same
    bf16 operands.  The accumulation term c 2^-24 sqrt(K) (|A| |B|^T) is the usual probabilistic bound of an fp32 sum
    of K products; bf16 outputs add the final rounding to 8 significant bits (at most 2^-8 relative)."""
    import torch
    K = A.shape[1]
    mag = A.double().abs() @ B.double().abs().t() * math.sqrt(K)
    if bias is not None:
        mag = mag + bias.double().abs()
    if resid is not None:
        mag = mag + resid.double().abs()
    bound = ELEM_C[kind] * 2.0 ** -24 * mag
    if kind == "bf16":
        bound = bound + BF16_OUT_ROUND * ref.abs()
    r = (out.double() - ref).abs() / bound.clamp_min(1e-300)
    r = torch.where(torch.isnan(r), torch.full_like(r, float("inf")), r)
    i = int(r.argmax())
    return {"elem_ratio": float(r.flatten()[i]), "elem_worst": [i // out.shape[1], i % out.shape[1]]}


# ------------------------------------------------------------------------------------------ gemm
def group_gemm(res):
    import torch
    from mudpt_b200 import _lib
    lib = _lib.load()
    dev = torch.device("cuda")
    st = _lib.stream_ptr(dev)
    torch.manual_seed(0)

    def guarded(rows, N, dtype):
        # NaN everywhere (an element the kernel fails to write fails its block) and GUARD rows after the output
        big = torch.full((rows + GUARD, N), float("nan"), device=dev, dtype=dtype)
        return big, big[:rows]

    def run(M, N, K, mode, np_=4, L=7):
        A = (torch.randn(M, K, device=dev) * 0.5).bfloat16()
        B = (torch.randn(N, K, device=dev) * 0.5).bfloat16()
        bias = torch.randn(N, device=dev)
        ref = A.double() @ B.double().t()  # exact products of the bf16 operands, fp64 sums
        kw = dict(out1=None, resid=None, aux=None, np_=1, L=1)
        bf, f32 = torch.bfloat16, torch.float32
        if mode == 0:
            big, out = guarded(M, N, bf); exp = ref + bias.double()
        elif mode == 1:
            big, out = guarded(M, N, f32); exp = ref + bias.double()
        elif mode == 2:
            resid = torch.randn(M, N, device=dev); kw["resid"] = resid
            big, out = guarded(M, N, f32); exp = ref + bias.double() + resid.double()
        elif mode == 3:
            big, out = guarded(M, N, bf)
            big1, out1 = guarded(M, N, bf); kw["out1"] = out1
            h = ref + bias.double(); exp = h
        elif mode == 4:
            aux = torch.randn(M, N, device=dev).bfloat16(); kw["aux"] = aux
            big, out = guarded(M, N, bf)
            hf = aux.double(); s = torch.sigmoid(1.702 * hf)
            exp = (ref + bias.double()) * (s * (1 + 1.702 * hf * (1 - s)))
        elif mode == 5:
            assert M % np_ == 0
            pos = torch.randn(np_ + 1, N, device=dev); kw["resid"] = pos; kw["np_"] = np_; kw["L"] = L
            big, out = guarded(M // np_ * L, N, f32)
            r = torch.arange(M, device=dev)
            dst = (r // np_) * L + 1 + r % np_
            exp = ref + bias.double() + pos.double()[1 + r % np_]
        rc = lib.mudpt_gemm_bf16(A.data_ptr(), B.data_ptr(), M, N, K, mode, out.data_ptr(),
                                 kw["out1"].data_ptr() if kw["out1"] is not None else None, bias.data_ptr(),
                                 kw["resid"].data_ptr() if kw["resid"] is not None else None,
                                 kw["aux"].data_ptr() if kw["aux"] is not None else None, N, kw["np_"], kw["L"], st)
        _lib.check(rc)
        torch.cuda.synchronize()
        if mode == 5:
            # rows r % L == 0 (CLS) and r % L > np_ (prompt slots) belong to other writers: they must keep the sentinel
            m = _metrics(out[dst], exp, tile=GEMM_TILE)
            other = torch.ones(out.shape[0], dtype=torch.bool, device=dev)
            other[dst] = False
            m["untouched"] = bool(torch.isnan(out[other]).all())
        else:
            m = _metrics(out, exp, tile=GEMM_TILE)
        if mode in (0, 1, 2):
            m.update(_gemm_elementwise(out, exp, A, B, "bf16" if mode == 0 else "f32", bias=bias, resid=kw["resid"]))
        if mode == 3:
            m2 = _metrics(out1, exp * torch.sigmoid(1.702 * exp), tile=GEMM_TILE)
            m["gelu_rel"], m["gelu_blk_rel"], m["gelu_blk_worst"] = m2["rel"], m2["blk_rel"], m2["blk_worst"]
            m["guards_intact"] = bool(torch.isnan(big[-GUARD:]).all() and torch.isnan(big1[-GUARD:]).all())
        else:
            m["guards_intact"] = bool(torch.isnan(big[-GUARD:]).all())
        return m

    shapes = [(128, 128, 64), (128, 128, 256), (128, 256, 64), (256, 512, 128), (6368, 2304, 768), (6368, 768, 3072),
              (900, 1536, 512), (77, 64, 64), (300, 136, 200), (21, 384, 128), (784, 768, 592),
              # strip-scheduler stress: ragged N (not a multiple of 32 / 256), M tails in both tile engines
              (4000, 1544, 256), (9625, 520, 128), (513, 96, 64), (2500, 40, 64),
              # long-K N = d shapes whose tile count is just above whole waves (75 / 76 pair tiles on 74 pairs)
              (9625, 512, 2048), (6368, 768, 2304), (19000, 768, 1024)]
    all_modes = [(128, 128, 64), (6368, 2304, 768), (300, 136, 200), (4000, 1544, 256), (9625, 520, 128),
                 (9625, 512, 2048), (6368, 768, 3072)]
    for (M, N, K) in shapes:
        for mode in ([0, 1, 2, 3, 4] if (M, N, K) in all_modes else [0]):
            key = f"gemm_{M}x{N}x{K}_m{mode}"
            try:
                res[key] = run(M, N, K, mode)
            except Exception as e:  # noqa
                res[key] = {"error": repr(e)}
                raise
            print(key, res[key], flush=True)
    res["gemm_patch_m5"] = run(4 * 6, 128, 768, 5)
    print("gemm_patch_m5", res["gemm_patch_m5"], flush=True)
    # the stems of the towers (B images x np patches, L = 1 + np + 2 prompt rows): ViT-B/16 at B = 32 (pair tiles) and
    # B = 165, ViT-B/32 (K = 3072), ViT-L/14 at B = 8 (Kp = 592: a K tail of 16)
    for (M, N, K, np_, L) in [(6272, 768, 768, 196, 199), (32340, 768, 768, 196, 199), (1568, 768, 3072, 49, 52),
                              (2048, 1024, 592, 256, 259)]:
        key = f"gemm_patch_{M}x{N}x{K}_m5"
        res[key] = run(M, N, K, 5, np_, L)
        print(key, res[key], flush=True)
    # error pattern of the smallest case for debugging, if wrong
    m = res["gemm_128x128x64_m0"]
    res["gemm_ok"] = all(v.get("rel", 1) < 2e-2 for k, v in res.items() if k.startswith("gemm_") and isinstance(v, dict))
    # timing of the big shapes
    import torch
    for (M, N, K) in [(6368, 2304, 768), (6368, 768, 768), (6368, 3072, 768), (6368, 768, 3072), (77000, 1536, 512)]:
        A = torch.randn(M, K, device=dev).bfloat16(); B = torch.randn(N, K, device=dev).bfloat16()
        out = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
        for _ in range(3):
            lib.mudpt_gemm_bf16(A.data_ptr(), B.data_ptr(), M, N, K, 0, out.data_ptr(), None, None, None, None, N, 1, 1, st)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            lib.mudpt_gemm_bf16(A.data_ptr(), B.data_ptr(), M, N, K, 0, out.data_ptr(), None, None, None, None, N, 1, 1, st)
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 10
        c = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
        for _ in range(3):
            torch.matmul(A, B.t(), out=c)
        e0.record()
        for _ in range(10):
            torch.matmul(A, B.t(), out=c)
        e1.record(); torch.cuda.synchronize()
        ms_t = e0.elapsed_time(e1) / 10
        res[f"gemm_time_{M}x{N}x{K}"] = {"ms": ms, "tflops": 2 * M * N * K / ms / 1e9, "cublas_ms": ms_t,
                                        "cublas_tflops": 2 * M * N * K / ms_t / 1e9}
        print(f"gemm_time_{M}x{N}x{K}", res[f"gemm_time_{M}x{N}x{K}"], flush=True)
    # the text-tower shapes of BASELINE config 2 with their real epilogues
    M = 77000
    for (N, K, mode, tag) in [(1536, 512, 0, "qkv"), (512, 512, 2, "out_proj+resid"), (2048, 512, 3, "c_fc+gelu"),
                              (512, 2048, 2, "c_proj+resid"), (2048, 512, 4, "d_c_proj*gelu'"), (512, 2048, 0, "d_c_fc")]:
        A = torch.randn(M, K, device=dev).bfloat16(); B = torch.randn(N, K, device=dev).bfloat16()
        bias = torch.randn(N, device=dev)
        f32 = mode in (1, 2)
        out = torch.empty(M, N, device=dev, dtype=torch.float32 if f32 else torch.bfloat16)
        out1 = torch.empty(M, N, device=dev, dtype=torch.bfloat16) if mode == 3 else None
        resid = torch.randn(M, N, device=dev) if mode == 2 else None
        aux = torch.randn(M, N, device=dev).bfloat16() if mode == 4 else None

        def call():
            lib.mudpt_gemm_bf16(A.data_ptr(), B.data_ptr(), M, N, K, mode, out.data_ptr(),
                                out1.data_ptr() if out1 is not None else None, bias.data_ptr(),
                                resid.data_ptr() if resid is not None else None,
                                aux.data_ptr() if aux is not None else None, N, 1, 1, st)
        for _ in range(3):
            call()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            call()
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 10
        nbytes = 2 * (M * K + N * K) + M * N * ((4 if f32 else 2) + (2 if mode == 3 else 0) + (4 if mode == 2 else 0) + (2 if mode == 4 else 0))
        res[f"gemm_text_{tag}"] = {"ms": ms, "tflops": 2 * M * N * K / ms / 1e9, "gbs": nbytes / ms / 1e6,
                                   "hbm_bound_ms": nbytes / 6538.3e6, "mma_bound_ms": 2 * M * N * K / 1618.5e9}
        print(f"gemm_text_{tag}", res[f"gemm_text_{tag}"], flush=True)


# ------------------------------------------------------------------------------------------ fused-LN GEMM modes, stream-K
def _row_stats_ref(x):
    """[M, d] fp32 -> [M, d/64, 2]: (sum, M2 about the span mean) per 64 columns, as rowstats / EPI_RESID_STATS emit."""
    import torch
    M, d = x.shape
    xs = x.double().view(M, d // 64, 64)
    return torch.stack([xs.sum(-1), ((xs - xs.mean(-1, keepdim=True)) ** 2).sum(-1)], -1).float().contiguous()


def _gemm_fused(lib, st, A, B, M, N, K, **kw):
    import ctypes as C
    from mudpt_b200 import _lib
    ep = _lib.GemmEpilogue()
    ep.ldc = N
    ep.ln_eps = 1e-5
    ep.splice_L = 1
    ep.stream_k = -1
    for k, v in kw.items():
        setattr(ep, k, v.data_ptr() if hasattr(v, "data_ptr") else v)
    _lib.check(lib.mudpt_gemm_fused(A.data_ptr(), B.data_ptr(), M, N, K, C.byref(ep), st))


def group_gemm_fused(res):
    import torch
    import torch.nn.functional as F
    from mudpt_b200 import _lib
    lib = _lib.load()
    dev = torch.device("cuda")
    st = _lib.stream_ptr(dev)
    torch.manual_seed(5)
    bf = torch.bfloat16

    def fold(W, gamma, beta, bias):
        N, K = W.shape
        Wl = torch.empty(N, K, device=dev, dtype=bf); Wlt = torch.empty(K, N, device=dev, dtype=bf)
        bl = torch.empty(N, device=dev); cs = torch.empty(N, device=dev); sb = torch.empty(N, 2, device=dev)
        _lib.check(lib.mudpt_fold_layernorm(W.data_ptr(), gamma.data_ptr(), beta.data_ptr(), bias.data_ptr(), Wl.data_ptr(),
                                            Wlt.data_ptr(), bl.data_ptr(), cs.data_ptr(), sb.data_ptr(), N, K, st))
        return Wl, Wlt, bl, cs, sb

    def prep(x):
        M, d = x.shape
        xb = torch.empty(M, d, device=dev, dtype=bf); stats = torch.empty(M, d // 64, 2, device=dev)
        _lib.check(lib.mudpt_rowstats(x.data_ptr(), xb.data_ptr(), stats.data_ptr(), M, d, st))
        return xb, stats

    def guarded(rows, *shape, dtype=torch.float32):
        # NaN everywhere (an element the kernel fails to write fails its block) and GUARD rows after the output
        big = torch.full((rows + GUARD, *shape), float("nan"), device=dev, dtype=dtype)
        return big, big[:rows]

    def intact(*bigs):
        return all(bool(torch.isnan(b[-GUARD:]).all()) for b in bigs)

    # ---- fold + rowstats
    W = torch.randn(384, 256, device=dev) * 0.06; gamma = 1 + 0.2 * torch.randn(256, device=dev)
    beta = 0.3 * torch.randn(256, device=dev); bias = torch.randn(384, device=dev)
    Wl, Wlt, bl, cs, sb = fold(W, gamma, beta, bias)
    torch.cuda.synchronize()
    res["fold"] = {"w_exact": bool(torch.equal(Wl, (W * gamma).to(bf))), "wt_exact": bool(torch.equal(Wlt, Wl.t().contiguous())),
                   "bias": _metrics(bl, bias + W @ beta), "colsum": _metrics(cs, Wl.float().sum(1)),
                   "sb_ok": bool(torch.equal(sb[:, 0], cs) and torch.equal(sb[:, 1], bl))}
    print("fold", res["fold"], flush=True)
    x = torch.randn(777, 768, device=dev) * 1.7 + 25.0  # a row mean far above the spread: M2 must not cancel
    xb, stats = prep(x)
    torch.cuda.synchronize()
    ref = _row_stats_ref(x)
    res["rowstats"] = {"xb_exact": bool(torch.equal(xb, x.to(bf))), "sum": _metrics(stats[..., 0], ref[..., 0]),
                       "m2": _metrics(stats[..., 1], ref[..., 1])}
    print("rowstats", res["rowstats"], flush=True)

    # ---- modes 7 / 8: LayerNorm + Linear (+ QuickGELU) in one GEMM
    for (M, N, K, shift, sk) in [(300, 384, 128, 0.0, -1), (6368, 2304, 768, 0.4, 1), (6368, 2304, 768, 0.4, 0),
                                 (9625, 1536, 512, 0.2, 1), (2000, 2048, 512, 3.0, -1), (130, 128, 64, 0.1, 1)]:
        x = torch.randn(M, K, device=dev) * 1.3 + shift
        x[:, 5] *= 8.0  # an outlier channel
        W = torch.randn(N, K, device=dev) * K ** -0.5; gamma = 1 + 0.2 * torch.randn(K, device=dev)
        beta = 0.2 * torch.randn(K, device=dev); bias = 0.5 * torch.randn(N, device=dev)
        Wl, Wlt, bl, cs, sb = fold(W, gamma, beta, bias)
        xb, stats = prep(x)
        exact = F.layer_norm(x.double(), (K,), gamma.double(), beta.double(), 1e-5) @ W.double().t() + bias.double()
        unfused = (F.layer_norm(x, (K,), gamma, beta, 1e-5).to(bf).float() @ W.to(bf).float().t() + bias).to(bf)
        um = _metrics(unfused, exact, tile=GEMM_TILE)
        ubase = dict(unfused_rel=um["rel"], unfused_blk_rel=um["blk_rel"])
        bigo, out = guarded(M, N, dtype=bf)
        _gemm_fused(lib, st, xb, Wl, M, N, K, mode=7, out0=out, bias=bl, colsum=cs, ln_stats=stats, ln_parts=K // 64, ln_width=K, stream_k=sk)
        torch.cuda.synchronize()
        key = f"gemmf_{M}x{N}x{K}_sk{sk}"
        res[key + "_m7"] = dict(_metrics(out, exact, tile=GEMM_TILE), **ubase, guards_intact=intact(bigo))
        bigh, h = guarded(M, N, dtype=bf); bigg, g = guarded(M, N, dtype=bf)
        _gemm_fused(lib, st, xb, Wl, M, N, K, mode=8, out0=h, out1=g, bias=bl, colsum=cs, ln_stats=stats, ln_parts=K // 64, ln_width=K, stream_k=sk)
        torch.cuda.synchronize()
        eg = exact * torch.sigmoid(1.702 * exact)
        gm = _metrics(g, eg, tile=GEMM_TILE)
        res[key + "_m8"] = dict(_metrics(h, exact, tile=GEMM_TILE), gelu_rel=gm["rel"], gelu_blk_rel=gm["blk_rel"],
                                gelu_blk_worst=gm["blk_worst"], **ubase, guards_intact=intact(bigh, bigg))
        print(key, res[key + "_m7"], res[key + "_m8"], flush=True)

    # ---- mode 9: residual + bf16 copy + statistics + splice
    for (M, N, K, L, row0, n, sk) in [(6368, 768, 3072, 199, 197, 2, 1), (6368, 768, 768, 199, 197, 2, 1), (9625, 512, 2048, 77, 1, 2, 1),
                                      (9625, 512, 512, 77, 1, 2, 0), (260, 128, 128, 13, 3, 4, 1), (1000, 1024, 256, 1, 0, 0, -1)]:
        A = (torch.randn(M, K, device=dev) * 0.5).to(bf); B = (torch.randn(N, K, device=dev) * 0.5).to(bf)
        bias = torch.randn(N, device=dev); resid = torch.randn(M, N, device=dev) * 3 + 1.5
        prompt = torch.randn(max(n, 1), N, device=dev)
        exp = A.double() @ B.double().t() + bias.double() + resid.double()
        if n > 0:
            rows = torch.arange(M, device=dev)
            pos = rows % L - row0
            sel = (pos >= 0) & (pos < n)
            exp[sel] = prompt.double()[pos[sel]]
        bigo, out = guarded(M, N); bigo2, out2 = guarded(M, N, dtype=bf)
        bigs, stats = guarded(M, N // 64, 2)
        _gemm_fused(lib, st, A, B, M, N, K, mode=9, out0=out, out2=out2, bias=bias, resid=resid, stats_out=stats,
                    splice_prompt=prompt if n > 0 else 0, splice_row0=row0, splice_n=n, splice_L=L, stream_k=sk)
        torch.cuda.synchronize()
        sref = _row_stats_ref(out)
        key = f"gemmf_{M}x{N}x{K}_sk{sk}_m9"
        res[key] = dict(_metrics(out, exp, tile=GEMM_TILE), out2_exact=bool(torch.equal(out2, out.to(bf))),
                        guards_intact=intact(bigo, bigo2, bigs),
                        splice_exact=bool(n == 0 or torch.equal(out[sel], prompt[pos[sel]])),
                        sum_rel=_metrics(stats[..., 0], sref[..., 0], tile=(128, N // 64))["blk_rel"],
                        m2_rel=_metrics(stats[..., 1], sref[..., 1], tile=(128, N // 64))["blk_rel"])
        print(key, res[key], flush=True)

    # ---- mode 11 -> mode 10: GELU' with row dots, then the LayerNorm dgrad in the dgrad GEMM's epilogue
    for (M, d, sk) in [(6368, 768, 1), (9625, 512, 1), (300, 128, 0), (2000, 512, -1)]:
        x = torch.randn(M, d, device=dev) * 1.4 + 0.3
        W = torch.randn(4 * d, d, device=dev) * d ** -0.5; gamma = 1 + 0.2 * torch.randn(d, device=dev)
        beta = 0.2 * torch.randn(d, device=dev); bias = 0.3 * torch.randn(4 * d, device=dev)
        Wl, Wlt, bl, cs, sb = fold(W, gamma, beta, bias)
        xb, stats = prep(x)
        # forward pre-activation h (bf16) as the fused forward saves it
        hsave = torch.zeros(M, 4 * d, device=dev, dtype=bf); gsave = torch.zeros(M, 4 * d, device=dev, dtype=bf)
        _gemm_fused(lib, st, xb, Wl, M, 4 * d, d, mode=8, out0=hsave, out1=gsave, bias=bl, colsum=cs, ln_stats=stats, ln_parts=d // 64, ln_width=d)
        dxo = (torch.randn(M, d, device=dev) * 0.1).to(bf)                    # gradient of the block output (bf16 copy)
        Wp_t = (torch.randn(4 * d, d, device=dev) * (4 * d) ** -0.5).to(bf)   # c_proj weight, transposed: [4d, d]
        span = int(lib.mudpt_gemm_dots_span(4 * d)); P = (4 * d + span - 1) // span
        bigdh, dh = guarded(M, 4 * d, dtype=bf); bigdots, dots = guarded(M, P, 2)
        _gemm_fused(lib, st, dxo, Wp_t, M, 4 * d, d, mode=11, out0=dh, aux=hsave, sb=sb, dots_out=dots, stream_k=sk)
        torch.cuda.synchronize()
        hf = hsave.float(); sg = torch.sigmoid(1.702 * hf)
        dh_ref = (dxo.float() @ Wp_t.float().t()) * (sg * (1 + 1.702 * hf * (1 - sg)))
        d1_ref = (dh_ref * cs).sum(1); d2_ref = (dh_ref * (hf - bl)).sum(1)
        key = f"gemmf_lnbwd_{M}x{d}_sk{sk}"
        # the row dots per 128-row band (one GEMM row tile)
        res[key + "_m11"] = dict(_metrics(dh, dh_ref, tile=GEMM_TILE), dot1=_metrics(dots[..., 0].sum(1, keepdim=True), d1_ref[:, None], tile=(128, 1)),
                                 dot2=_metrics(dots[..., 1].sum(1, keepdim=True), d2_ref[:, None], tile=(128, 1)), guards_intact=intact(bigdh, bigdots))
        # mode 10 against autograd through LayerNorm + Linear with the SAME dh
        for with_resid in (True, False):
            resid = torch.randn(M, d, device=dev) if with_resid else None
            bigdx, dx = guarded(M, d); bigdx16, dx16 = guarded(M, d, dtype=bf)
            if with_resid:
                dx.copy_(resid)
            _gemm_fused(lib, st, dh, Wlt, M, d, 4 * d, mode=10, out0=dx, out2=dx16, resid=dx if with_resid else 0, x2=xb,
                        ln_stats=stats, ln_parts=d // 64, ln_width=d, dots=dots, dot_parts=P, stream_k=sk)
            torch.cuda.synchronize()
            xr = x.double().clone().requires_grad_(True)
            y = F.layer_norm(xr, (d,), gamma.double(), beta.double(), 1e-5) @ W.double().t()
            y.backward(dh.double())
            exp = xr.grad + (resid.double() if with_resid else 0)
            res[key + f"_m10_r{int(with_resid)}"] = dict(_metrics(dx, exp, tile=GEMM_TILE), out2_exact=bool(torch.equal(dx16, dx.to(bf))),
                                                         guards_intact=intact(bigdx, bigdx16))
        print(key, res[key + "_m11"], res[key + "_m10_r1"], res[key + "_m10_r0"], flush=True)

    # ---- attention backward with the row dots of dqkv
    for (S, L, H, causal) in [(3, 199, 12, 0), (5, 77, 8, 1), (4, 9, 8, 1), (2, 130, 2, 1)]:
        d = H * 64
        qkv = torch.randn(S * L, 3 * d, device=dev).to(bf)
        o = torch.zeros(S * L, d, device=dev, dtype=bf); lse = torch.zeros(S, H, L, device=dev)
        _lib.check(lib.mudpt_attention_forward(qkv.data_ptr(), o.data_ptr(), lse.data_ptr(), S, L, H, causal, st))
        do = torch.randn(S * L, d, device=dev).to(bf)
        dqkv = torch.zeros(S * L, 3 * d, device=dev, dtype=bf); dsum = torch.zeros(S, H, L, device=dev)
        sb = torch.randn(3 * d, 2, device=dev); dots = torch.zeros(S * L, 3 * H, 2, device=dev)
        lib.mudpt_set_attention_tc(0)  # the row dots are a by-product of the warp-MMA kernels: compare like with like
        _lib.check(lib.mudpt_attention_backward_dots(qkv.data_ptr(), o.data_ptr(), do.data_ptr(), lse.data_ptr(), dsum.data_ptr(),
                                                     dqkv.data_ptr(), S, L, H, causal, sb.data_ptr(), dots.data_ptr(), st))
        dqkv2 = torch.zeros_like(dqkv)
        _lib.check(lib.mudpt_attention_backward(qkv.data_ptr(), o.data_ptr(), do.data_ptr(), lse.data_ptr(), dsum.data_ptr(),
                                                dqkv2.data_ptr(), S, L, H, causal, st))
        torch.cuda.synchronize()
        lib.mudpt_set_attention_tc(1)
        gq = dqkv.float().view(S * L, 3 * H, 64)
        d1 = (gq * sb[:, 0].view(3 * H, 64)).sum(-1)
        d2 = (gq * (qkv.float().view(S * L, 3 * H, 64) - sb[:, 1].view(3 * H, 64))).sum(-1)
        key = f"attn_dots_S{S}_L{L}_H{H}_c{causal}"
        res[key] = {"same_dqkv": bool(torch.equal(dqkv, dqkv2)), "dot1": _metrics(dots[..., 0], d1), "dot2": _metrics(dots[..., 1], d2)}
        print(key, res[key], flush=True)

    # ---- stream-K: equality with whole-tile scheduling + timing against cuBLAS on the shapes of the towers.
    # 24 back-to-back launches over 3 rotating operand / output sets per measurement (the CUDA event clock ticks in
    # ~2 us steps, and back-to-back launches with L2-warm activations are what the tower loop looks like).
    table = {}
    for (M, N, K) in [(6368, 2304, 768), (6368, 768, 768), (6368, 3072, 768), (6368, 768, 3072), (6368, 768, 2304),
                      (9625, 1536, 512), (9625, 512, 512), (9625, 2048, 512), (9625, 512, 2048), (9625, 512, 1536),
                      (77000, 1536, 512), (77000, 512, 2048), (77000, 512, 512), (250, 512, 2048), (2000, 512, 1536)]:
        As = [torch.randn(M, K, device=dev).to(bf) for _ in range(3)]
        B = torch.randn(N, K, device=dev).to(bf)
        outs_ = [torch.zeros(M, N, device=dev, dtype=bf) for _ in range(3)]
        ref = As[0].double() @ B.double().t()

        def timed(fn, reps=24):
            for i in range(3):
                fn(i)
            best = []
            for _ in range(3):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for i in range(reps):
                    fn(i)
                e1.record(); torch.cuda.synchronize()
                best.append(e0.elapsed_time(e1) / reps)
            return sorted(best)[1]

        outs, times = {}, {}
        for sk in (0, 1, -1):
            times[sk] = timed(lambda i: _gemm_fused(lib, st, As[i % 3], B, M, N, K, mode=0, out0=outs_[i % 3], stream_k=sk))
            outs_[0].fill_(float("nan"))  # the checked call starts from the sentinel
            _gemm_fused(lib, st, As[0], B, M, N, K, mode=0, out0=outs_[0], stream_k=sk)
            torch.cuda.synchronize()
            outs[sk] = outs_[0].clone()
        t_cublas = timed(lambda i: torch.matmul(As[i % 3], B.t(), out=outs_[i % 3]))
        fl = 2.0 * M * N * K / 1e9
        table[f"{M}x{N}x{K}"] = {"us_whole": round(times[0] * 1e3, 1), "us_streamk": round(times[1] * 1e3, 1),
                                 "us_auto": round(times[-1] * 1e3, 1), "us_cublas": round(t_cublas * 1e3, 1),
                                 "tflops_whole": round(fl / times[0], 0), "tflops_streamk": round(fl / times[1], 0),
                                 "tflops_auto": round(fl / times[-1], 0), "tflops_cublas": round(fl / t_cublas, 0),
                                 "max_abs_sk_vs_whole": float((outs[1].float() - outs[0].float()).abs().max())}
        for sk, sched in ((0, "whole"), (1, "streamk"), (-1, "auto")):
            m = _metrics(outs[sk], ref, tile=GEMM_TILE)
            table[f"{M}x{N}x{K}"].update({f"rel_{sched}": m["rel"], f"blk_rel_{sched}": m["blk_rel"], f"blk_worst_{sched}": m["blk_worst"]})
        del ref
        print("gemm_time", f"{M}x{N}x{K}", table[f"{M}x{N}x{K}"], flush=True)
    res["gemm_time_table"] = table


# ------------------------------------------------------------------------------------------ rowops
def group_rowops(res):
    import torch
    import torch.nn.functional as F
    from mudpt_b200 import _lib
    lib = _lib.load()
    dev = torch.device("cuda")
    st = _lib.stream_ptr(dev)
    torch.manual_seed(1)
    for (M, d) in [(37, 64), (1000, 512), (6368, 768), (513, 1024)]:
        x = torch.randn(M, d, device=dev) * 2 + 0.5
        g = torch.randn(d, device=dev); b = torch.randn(d, device=dev)
        ref = F.layer_norm(x.double(), (d,), g.double(), b.double(), 1e-5)
        o16 = torch.full((M, d), float("nan"), device=dev, dtype=torch.bfloat16)
        _lib.check(lib.mudpt_layernorm_forward(x.data_ptr(), g.data_ptr(), b.data_ptr(), o16.data_ptr(), 1, M, d, st))
        o32 = torch.full((M, d), float("nan"), device=dev)
        _lib.check(lib.mudpt_layernorm_forward(x.data_ptr(), g.data_ptr(), b.data_ptr(), o32.data_ptr(), 0, M, d, st))
        torch.cuda.synchronize()
        res[f"ln_fwd_{M}x{d}"] = {"f32": _metrics(o32, ref, grid=(M,)), "bf16": _metrics(o16, ref, grid=(M,))}
        xr = x.double().requires_grad_(True)
        dy = torch.randn(M, d, device=dev)
        resid = torch.randn(M, d, device=dev)
        F.layer_norm(xr, (d,), g.double(), b.double(), 1e-5).backward(dy.double())
        exp = resid.double() + xr.grad
        dx = resid.clone(); dx16 = torch.full((M, d), float("nan"), device=dev, dtype=torch.bfloat16)
        _lib.check(lib.mudpt_layernorm_backward(dy.data_ptr(), x.data_ptr(), g.data_ptr(), dx.data_ptr(), dx.data_ptr(),
                                                dx16.data_ptr(), M, d, st))
        torch.cuda.synchronize()
        res[f"ln_bwd_{M}x{d}"] = {"f32": _metrics(dx, exp, grid=(M,)), "bf16": _metrics(dx16, exp, grid=(M,))}
        print(f"ln_{M}x{d}", res[f"ln_fwd_{M}x{d}"], res[f"ln_bwd_{M}x{d}"], flush=True)
    # LayerNorm backward on the bf16 gradient stream (option grad_stream_bf16): bf16 dy, x as fp32 rows or bf16 + statistics,
    # residual gradient fp32 or bf16 IN PLACE (aliasing the bf16 output), fp32 rows written in the prompt window only
    def ln_bwd_ref(dy16, x_used, mean, rstd, gam, resid):
        xh = (x_used - mean) * rstd
        gg = dy16.float() * gam
        return resid + rstd * (gg - gg.mean(1, keepdim=True) - xh * (gg * xh).mean(1, keepdim=True))
    for (S_, L_, row0_, n_, d) in [(13, 77, 1, 2, 512), (32, 199, 197, 2, 768), (5, 9, 1, 4, 64), (3, 259, 257, 2, 1024)]:
        M = S_ * L_
        x = torch.randn(M, d, device=dev) * 2 + 0.5
        gam = torch.randn(d, device=dev)
        dy16 = torch.randn(M, d, device=dev).bfloat16()
        mean = x.mean(1, keepdim=True)
        rstd = torch.rsqrt(x.var(1, unbiased=False, keepdim=True) + 1e-5)
        xb = torch.empty(M, d, device=dev, dtype=torch.bfloat16)
        stats = torch.empty(M, d // 64, 2, device=dev)
        _lib.check(lib.mudpt_rowstats(x.data_ptr(), xb.data_ptr(), stats.data_ptr(), M, d, st))
        resid32 = torch.randn(M, d, device=dev)
        resid16 = resid32.bfloat16()
        tok = torch.arange(M, device=dev) % L_
        inwin = (tok >= row0_) & (tok < row0_ + n_)
        out = {}
        for xform in ("f32", "bf16"):
            x_used = x if xform == "f32" else xb.float()
            xp, sp = (x.data_ptr(), None) if xform == "f32" else (xb.data_ptr(), stats.data_ptr())
            for rform in ("f32", "bf16", "none"):
                resid = {"f32": resid32, "bf16": resid16.float(), "none": torch.zeros_like(resid32)}[rform]
                exp = ln_bwd_ref(dy16, x_used, mean, rstd, gam, resid)
                for win in (-1, n_, 0):
                    # outputs sit between guard bands of 8 rows (compute-sanitizer is closed on the GPU pool: a write outside
                    # the M rows -- e.g. from the last, partial 8-row block of the pipeline kernel -- shows up here)
                    big32 = torch.full((M + 16, d), 7.0, device=dev)
                    big16 = torch.full((M + 16, d), 3.0, device=dev, dtype=torch.bfloat16)
                    dx, dxb = big32[8:8 + M], big16[8:8 + M]
                    dxb.copy_(resid16)  # the bf16 residual is updated in place
                    rp = {"f32": resid32.data_ptr(), "bf16": dxb.data_ptr(), "none": None}[rform]
                    _lib.check(lib.mudpt_layernorm_backward_stream(dy16.data_ptr(), xp, sp, gam.data_ptr(), rp, 1 if rform == "bf16" else 0,
                                                                   dx.data_ptr(), dxb.data_ptr(), M, d, L_, row0_, win, st))
                    torch.cuda.synchronize()
                    wr = torch.ones_like(inwin) if win < 0 else (inwin if win > 0 else torch.zeros_like(inwin))
                    m = {"bf16": _metrics(dxb, exp, grid=(M,)),
                         "bf16_is_rounded_f32": bool(torch.equal(dxb[wr], dx[wr].bfloat16())),
                         "untouched": bool((dx[~wr] == 7.0).all()),
                         "guards_intact": bool((big32[:8] == 7.0).all() and (big32[8 + M:] == 7.0).all() and
                                               (big16[:8] == 3.0).all() and (big16[8 + M:] == 3.0).all())}
                    if bool(wr.any()):
                        m["f32"] = _metrics(dx[wr], exp[wr], grid=(int(wr.sum()),))
                    out[f"{xform}_{rform}_{win}"] = m
        # fp32 output not requested at all
        big16 = torch.full((M + 16, d), 3.0, device=dev, dtype=torch.bfloat16)
        dxb = big16[8:8 + M]
        dxb.copy_(resid16)
        _lib.check(lib.mudpt_layernorm_backward_stream(dy16.data_ptr(), xb.data_ptr(), stats.data_ptr(), gam.data_ptr(), dxb.data_ptr(), 1,
                                                       None, dxb.data_ptr(), M, d, L_, row0_, n_, st))
        torch.cuda.synchronize()
        out["no_f32"] = {"bf16": _metrics(dxb, ln_bwd_ref(dy16, xb.float(), mean, rstd, gam, resid16.float()), grid=(M,)),
                         "guards_intact": bool((big16[:8] == 3.0).all() and (big16[8 + M:] == 3.0).all())}
        res[f"ln_bwd_stream_{M}x{d}"] = out
        worst32 = max(v["f32"]["blk_rel"] for v in out.values() if "f32" in v)
        worst16 = max(v["bf16"]["blk_rel"] for v in out.values())
        print(f"ln_bwd_stream_{M}x{d}: worst fp32 row rel {worst32:.2e}, worst bf16 row rel {worst16:.2e}, "
              f"untouched {all(v.get('untouched', True) for v in out.values())}", flush=True)
    # splice
    S, L, row0, n, d = 33, 21, 19, 2, 768
    x = torch.randn(S, L, d, device=dev); p = torch.randn(n, d, device=dev)
    exp = x.clone(); exp[:, row0:row0 + n] = p
    _lib.check(lib.mudpt_splice_forward(x.data_ptr(), p.data_ptr(), S, L, row0, n, d, st))
    torch.cuda.synchronize()
    res["splice_fwd_bitexact"] = bool(torch.equal(x, exp))
    dx = torch.randn(S, L, d, device=dev); dx16 = dx.bfloat16().contiguous()
    exp_dp = dx[:, row0:row0 + n].double().sum(0).float()
    exp_dx = dx.clone(); exp_dx[:, row0:row0 + n] = 0
    dp = torch.full((n, d), float("nan"), device=dev)
    _lib.check(lib.mudpt_splice_backward(dx.data_ptr(), dx16.data_ptr(), dp.data_ptr(), S, L, row0, n, d, 1, st))
    torch.cuda.synchronize()
    res["splice_bwd"] = {"dp": _metrics(dp, exp_dp, grid=(n,)), "dx_zeroed": bool(torch.equal(dx, exp_dx)),
                         "dx16_zeroed": bool((dx16[:, row0:row0 + n] == 0).all())}
    print("splice", res["splice_fwd_bitexact"], res["splice_bwd"], flush=True)
    # im2col
    for (B, R, p_) in [(3, 224, 16), (2, 224, 14), (2, 32, 16)]:
        img = torch.randn(B, 3, R, R, device=dev)
        k = 3 * p_ * p_; ld = (k + 7) // 8 * 8
        gw = R // p_
        out = torch.zeros(B * gw * gw, ld, device=dev, dtype=torch.bfloat16)
        _lib.check(lib.mudpt_im2col(img.data_ptr(), out.data_ptr(), B, R, p_, ld, st))
        torch.cuda.synchronize()
        exp = F.unfold(img, kernel_size=p_, stride=p_).transpose(1, 2).reshape(B * gw * gw, k).bfloat16()
        res[f"im2col_{B}_{R}_{p_}"] = bool(torch.equal(out[:, :k], exp))
        print(f"im2col_{B}_{R}_{p_}", res[f"im2col_{B}_{R}_{p_}"], flush=True)


# ------------------------------------------------------------------------------------------ attention
def _attn_ref(qkv, S, L, H, causal):
    import torch
    d = H * 64
    q, k, v = qkv.view(S, L, 3, H, 64).permute(2, 0, 3, 1, 4)
    s = (q @ k.transpose(-1, -2)) * 0.125
    if causal:
        s = s + torch.full((L, L), float("-inf"), device=qkv.device, dtype=s.dtype).triu_(1)
    p = torch.softmax(s, -1)
    o = (p @ v).permute(0, 2, 1, 3).reshape(S * L, d)
    return o


# Longest sequence whose backward the short-sequence kernels take; they form D = rowsum(P dP) from the recomputed P.
# Longer sequences (both kernel families) read D = rowsum(dO O) from the bf16 O the forward stored.
ATTN_SHORT_MAX_L = 128


def _attn_emul_bf16(qkv, do, S, L, H, causal, o_stored=None):
    """(o, dq, dk, dv), bf16, of attention computed in fp32 with the kernels' roundings: P and dS rounded to bf16 as MMA
    operands, D = rowsum(P dP) or, past ATTN_SHORT_MAX_L, rowsum(dO O) with O the bf16 output the backward is given
    (`o_stored`, else this function's own).  The error this makes against fp64 is what a correct kernel of that design
    makes on the same inputs, problem by problem."""
    import torch
    d = H * 64
    q, k, v = qkv.float().view(S, L, 3, H, 64).permute(2, 0, 3, 1, 4)
    dO = do.float().view(S, L, H, 64).permute(0, 2, 1, 3)
    s = (q @ k.transpose(-1, -2)) * 0.125
    if causal:
        s = s + torch.full((L, L), float("-inf"), device=qkv.device).triu_(1)
    p = torch.softmax(s, -1)
    pb = p.bfloat16().float()
    o = (pb @ v).bfloat16().float()
    dP = dO @ v.transpose(-1, -2)
    if L <= ATTN_SHORT_MAX_L:
        D = (p * dP).sum(-1, keepdim=True)
    else:
        ob = o if o_stored is None else o_stored.float().view(S, L, H, 64).permute(0, 2, 1, 3)
        D = (dO * ob).sum(-1, keepdim=True)
    dS = (p * (dP - D)).bfloat16().float()
    dq, dk, dv = (dS @ k) * 0.125, (dS.transpose(-1, -2) @ q) * 0.125, pb.transpose(-1, -2) @ dO
    flat = lambda t: t.permute(0, 2, 1, 3).reshape(S * L, d).bfloat16()  # noqa: E731
    return flat(o), flat(dq), flat(dk), flat(dv)


def _attn_lse2_ref(qkv, S, L, H, causal):
    """[S, H, L] log2 of sum_j exp(q_i k_j / 8) over the visible keys (the kernels' lse2), from fp64 scores."""
    import torch
    q, k, _ = qkv.double().view(S, L, 3, H, 64).permute(2, 0, 3, 1, 4)
    s = (q @ k.transpose(-1, -2)) * 0.125
    if causal:
        s = s + torch.full((L, L), float("-inf"), device=qkv.device, dtype=s.dtype).triu_(1)
    return torch.logsumexp(s, -1) * (1.0 / math.log(2.0))


def _attn_peaked_qkv(S, L, H, kind, dev):
    """bf16 qkv whose softmax rows are far from flat.  "peak": q and k scaled by sqrt(8), score std ~ 8, a few keys
    carry each row.  "sink": every query shares a component u with key 0 (per head), which takes ~99 % of each row's
    mass, as the SOT / CLS tokens do in trained CLIP towers."""
    import torch
    qkv = torch.randn(S, L, 3, H, 64, device=dev)
    if kind == "peak":
        qkv[:, :, :2] *= math.sqrt(8.0)
    else:
        u = torch.randn(H, 64, device=dev)
        qkv[:, :, 0] += u
        qkv[:, 0, 1] = 1.5 * u
    return qkv.reshape(S * L, 3 * H * 64).bfloat16()


def _attn_blocks(t, S, L, H):
    """[S*L, H*64] (or [S, H, L]) -> [S, H, -1]: one block per (sequence, head) problem."""
    if t.dim() == 3:
        return t
    return t.reshape(S, L, H, -1).permute(0, 2, 1, 3)


def group_attention(res):
    import torch
    from mudpt_b200 import _lib
    lib = _lib.load()
    dev = torch.device("cuda")
    st = _lib.stream_ptr(dev)
    torch.manual_seed(2)
    shapes = [(3, 199, 12, 0), (5, 77, 8, 1), (7, 9, 8, 1), (4, 16, 2, 1), (2, 64, 1, 0), (2, 259, 16, 0),
              (3, 7, 2, 0), (2, 130, 2, 1)]
    # tile-boundary lengths of the short-sequence kernels (1 / 2 / 5 / 8 tiles, both masks) and the first
    # lengths that fall back to the generic ones
    shapes += [(2, L, 2, c) for L in (2, 15, 17, 31, 32, 33, 48, 79, 80, 81, 96, 127, 128, 129, 144) for c in (0, 1)]
    # the resident two-block tcgen05 backward: 3 / 4 query chunks, every tail width, more problems than SMs
    shapes += [(2, L, 2, c) for L in (145, 160, 176, 192, 193, 208, 224, 241, 255, 256) for c in (0, 1)]
    shapes += [(16, 199, 12, 0), (9, 197, 20, 0)]
    cases = [(S, L, H, c, None) for (S, L, H, c) in shapes]
    # peaked softmax rows at the towers' lengths: vision (199), text (77, EOT-truncated 9), ViT-L vision (259)
    cases += [(S, L, H, c, kind) for (S, L, H, c) in [(4, 199, 12, 0), (8, 77, 8, 1), (8, 9, 8, 1), (2, 259, 16, 0)]
              for kind in ("peak", "sink")]
    for (S, L, H, causal, kind) in cases:
        d = H * 64
        qkv = torch.randn(S * L, 3 * d, device=dev).bfloat16() if kind is None else _attn_peaked_qkv(S, L, H, kind, dev)
        do = torch.randn(S * L, d, device=dev).bfloat16()
        # fp64 reference on the same bf16 inputs
        qr = qkv.double().requires_grad_(True)
        oref = _attn_ref(qr, S, L, H, causal)
        oref.backward(do.double())
        g, oref = qr.grad, oref.detach()
        lse_ref = _attn_lse2_ref(qkv, S, L, H, causal)

        def blk(x, ref):
            return _metrics(_attn_blocks(x, S, L, H), _attn_blocks(ref, S, L, H), grid=(S, H))

        def forward(tc_mode):
            o = torch.full((S * L, d), float("nan"), device=dev, dtype=torch.bfloat16)
            lse = torch.full((S, H, L), float("nan"), device=dev)
            lib.mudpt_set_attention_tc(tc_mode)
            _lib.check(lib.mudpt_attention_forward(qkv.data_ptr(), o.data_ptr(), lse.data_ptr(), S, L, H, causal, st))
            torch.cuda.synchronize()
            lib.mudpt_set_attention_tc(1)
            return o, lse

        def backward(tc_mode, o, lse):
            dqkv = torch.full((S * L, 3 * d), float("nan"), device=dev, dtype=torch.bfloat16)
            dsum = torch.zeros(S, H, L, device=dev)
            lib.mudpt_set_attention_tc(tc_mode)
            _lib.check(lib.mudpt_attention_backward(qkv.data_ptr(), o.data_ptr(), do.data_ptr(), lse.data_ptr(), dsum.data_ptr(),
                                                    dqkv.data_ptr(), S, L, H, causal, st))
            torch.cuda.synchronize()
            lib.mudpt_set_attention_tc(1)
            grads[tc_mode] = dqkv
            return {"dq": blk(dqkv[:, :d], g[:, :d]), "dk": blk(dqkv[:, d:2 * d], g[:, d:2 * d]), "dv": blk(dqkv[:, 2 * d:], g[:, 2 * d:])}

        grads = {}
        o, lse = forward(0)  # warp-MMA kernels
        r = {"o": blk(o, oref), "lse": blk(lse, lse_ref)}
        tc = {}
        if L <= 256:  # tcgen05 / TMEM kernels on the same input: output and log-sum-exp (the backward below uses them)
            o_w, lse_w = o, lse
            o, lse = forward(2)
            tc = {"o_warp": r["o"], "lse_warp": r["lse"], "lse_vs_warp": _metrics(lse, lse_w)}
            r["o"], r["lse"] = blk(o, oref), blk(lse, lse_ref)
        r.update(backward(0, o, lse))
        tc.update(backward(2, o, lse))  # tcgen05 backward (both launches) on the same input, any length
        r["tc"] = tc
        key = f"attn_S{S}_L{L}_H{H}_c{causal}"
        if kind is not None:
            # the same computation in fp32 with the kernels' roundings: the error a correct kernel of this design makes on
            # these rows (dS = P (dP - D) cancels on peaked rows)
            oe, dqe, dke, dve = _attn_emul_bf16(qkv, do, S, L, H, causal, o_stored=o)
            r["emul"] = {"o": blk(oe, oref), "dq": blk(dqe, g[:, :d]), "dk": blk(dke, g[:, d:2 * d]), "dv": blk(dve, g[:, 2 * d:])}
            # every problem's error (row-major over (sequence, head)), kernel and emulation, for a block-by-block bound
            for i, (part, em) in enumerate((("dq", dqe), ("dk", dke), ("dv", dve))):
                gb_ = _attn_blocks(g[:, i * d:(i + 1) * d], S, L, H)
                r["emul"][part]["blk_all"] = _block_rel(_attn_blocks(em, S, L, H), gb_, grid=(S, H)).tolist()
                for tc_mode, dst in ((0, r), (2, tc)):
                    kb = _attn_blocks(grads[tc_mode][:, i * d:(i + 1) * d], S, L, H)
                    dst[part]["blk_all"] = _block_rel(kb, gb_, grid=(S, H)).tolist()
            key += f"_{kind}"
        res[key] = r
        print(key, {p: (round(v["rel"], 6), round(v["blk_rel"], 6), v["blk_worst"]) for p, v in r.items() if "blk_rel" in v},
              {p: round(v["blk_rel"], 6) for p, v in tc.items() if "blk_rel" in v},
              {p: round(v["blk_rel"], 6) for p, v in r.get("emul", {}).items()}, flush=True)
    # timing at the cfg-2 shapes: vision, full-length text, EOT-truncated text
    for (S, L, H, causal, tag) in [(32, 199, 12, 0, "vision"), (1000, 77, 8, 1, "text77"), (1000, 9, 8, 1, "text9")]:
        for mode in (0, 2):
            lib.mudpt_set_attention_tc(mode)
            _time_attention(res, lib, st, dev, S, L, H, causal, tag + ("_tc" if mode else "_warp"))
    lib.mudpt_set_attention_tc(1)


def _time_attention(res, lib, st, dev, S, L, H, causal, tag):
    import torch
    if True:
        d = H * 64
        qkv = torch.randn(S * L, 3 * d, device=dev).bfloat16()
        o = torch.zeros(S * L, d, device=dev, dtype=torch.bfloat16); lse = torch.zeros(S, H, L, device=dev)
        do = torch.randn(S * L, d, device=dev).bfloat16(); dqkv = torch.zeros(S * L, 3 * d, device=dev, dtype=torch.bfloat16)
        dsum = torch.zeros(S, H, L, device=dev)
        for name, fn in [("fwd", lambda: lib.mudpt_attention_forward(qkv.data_ptr(), o.data_ptr(), lse.data_ptr(), S, L, H, causal, st)),
                         ("bwd", lambda: lib.mudpt_attention_backward(qkv.data_ptr(), o.data_ptr(), do.data_ptr(), lse.data_ptr(),
                                                                      dsum.data_ptr(), dqkv.data_ptr(), S, L, H, causal, st))]:
            for _ in range(3):
                fn()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(20):
                fn()
            e1.record(); torch.cuda.synchronize()
            us = e0.elapsed_time(e1) / 20 * 1e3
            nbytes = S * L * d * 2 * (4 if name == "fwd" else 8)
            res[f"attn_time_{tag}_{name}_us"] = us
            print(f"attn_time_{tag}_{name}_us", round(us, 1), "hbm-bound us", round(nbytes / 6538.3e3, 1), flush=True)


# ------------------------------------------------------------------------------------------ head + model
def _compare_model(name, res, fused=True):
    import torch
    import torch.nn.functional as F
    from tests import golden_util as gu
    from oracle import mudpt_oracle as orc
    c = gu.load(name)
    g = c["golden"]
    model, _ = gu.build_model(c, "cuda")
    image, labels = c["image"].cuda(), c["labels"].cuda()
    out = {}
    for mode in (["fused", "autograd"] if fused else ["autograd"]):
        model.zero_grad(set_to_none=True)
        if mode == "fused":
            loss, logits = model.forward_backward(image, labels)
        else:
            logits = model(image)
            loss = F.cross_entropy(logits, labels)
            loss.backward()
        torch.cuda.synchronize()
        r = {"loss": float(loss), "loss_ref": float(g["loss"]),
             "logits": _metrics(logits.detach().cpu(), torch.from_numpy(g["logits"]))}
        ref_logits = torch.from_numpy(g["logits"])
        r["top1"] = orc.top1_agreement(logits.detach().cpu(), ref_logits, r["logits"]["max_abs"])
        for k in orc.TRAINABLE:
            p = dict(model.named_parameters())[k]
            ref = torch.from_numpy(g["grad/" + k])
            if ref.numel() and float(ref.norm()) > 0:
                r["grad/" + k] = _metrics(p.grad.detach().cpu(), ref)
        out[mode] = r
        print(name, mode, json.dumps(r), flush=True)
    # features through the module-level API
    with torch.no_grad():
        prompts, shared, text_deep, t2v = model.mudpt_prompt_learner()
        f_img, v2t = model.image_encoder(image, shared, t2v)
        f_txt = model.text_encoder(prompts, model.tokenized_prompts, text_deep + v2t)
    out["image_features"] = _metrics(f_img.cpu(), torch.from_numpy(g["image_features"]))
    out["text_features"] = _metrics(f_txt.cpu(), torch.from_numpy(g["text_features"]))
    print(name, "features", out["image_features"], out["text_features"], flush=True)
    # truncated vs full-length text tower (exact under the causal mask)
    model.truncate_text_to_eot = False
    with torch.no_grad():
        lf = model(image)
    out["full_len_logits"] = _metrics(lf.cpu(), torch.from_numpy(g["logits"]))
    print(name, "full-length logits", out["full_len_logits"], flush=True)
    res[name] = out


def _head_engine(e, dev, vision_width=128, layers=1):
    """A native handle whose text width = embed_dim = e (the logits head takes its width from the handle)."""
    from mudpt_b200.engine import Engine
    from mudpt_b200 import synthetic as syn
    arch = dict(zip(["embed_dim", "image_resolution", "vision_layers", "vision_width", "vision_patch_size", "context_length",
                     "vocab_size", "transformer_width", "transformer_heads", "transformer_layers"], syn.ARCHS["tiny"].astuple()))
    arch.update(embed_dim=e, transformer_width=e, transformer_heads=e // 64, vision_width=vision_width,
                vision_layers=layers, transformer_layers=layers)
    return Engine(arch, 2, 1, dev)


def group_head(res):
    import torch
    import torch.nn.functional as F
    from mudpt_b200 import _lib
    dev = torch.device("cuda")
    st = _lib.stream_ptr(dev)
    torch.manual_seed(3)
    # logits / cross-entropy head at the embed widths of ViT-B/16 (512) and ViT-L/14 (768) and at 64; logit scales of a
    # fresh CLIP (1 / 0.07) and of trained weights (100); the loss scale of one rank of eight (inv_global_batch = 1 / 8B).
    # (64, 1000) at 768 reads image rows from L2 in head_cols_kernel (b_smem < B); (4, 70000) takes the unfused path
    # (l2norm / split-K sgemm / ce_rows_kernel); C < 8 leaves cluster slices empty; (256, 1000) is the logits-only call.
    cases = {64: [(4, 10), (32, 1000)],
             512: [(1, 1), (7, 9), (32, 125), (32, 1000), (32, 1001), (256, 1000)],
             768: [(1, 1), (7, 9), (32, 125), (32, 1000), (32, 1001), (64, 1000), (4, 70000), (256, 1000)]}
    for e, shapes in cases.items():
        eng = _head_engine(e, dev)
        for ls_name, ls_val in (("clip", math.log(1 / 0.07)), ("trained", math.log(100.0))):
            ls = torch.tensor(ls_val, device=dev)
            _lib.check(eng.lib.mudpt_set_weight(eng.h, b"logit_scale", ls.data_ptr(), 1, st), eng.h)
            torch.cuda.synchronize()
            scale = math.exp(ls_val)
            for (B, Cn) in shapes:
                logits_only = (B, Cn) == (256, 1000)
                igb = 1.0 / (8 * B)
                fi = torch.randn(B, e, device=dev) * 0.3
                ft = torch.randn(Cn, e, device=dev) * 0.3
                y = torch.randint(0, Cn, (B,), device=dev)
                y[0] = 0
                y[-1] = Cn - 1
                fid, ftd = fi.double().requires_grad_(True), ft.double().requires_grad_(True)
                logits_ref = scale * F.normalize(fid, dim=-1) @ F.normalize(ftd, dim=-1).t()
                key = f"logits_head_e{e}_{B}x{Cn}_{ls_name}"
                r = {}
                if logits_only:
                    logits, _, _, _ = eng.logits_head(fi, ft, None, igb, False)
                    torch.cuda.synchronize()
                    r["logits"] = _metrics(logits, logits_ref.detach(), grid=(B,))
                    r["logits_cols"] = _metrics(logits.t(), logits_ref.detach().t(), grid=(Cn,))
                    res[key] = r
                    print(key, {p: (v["blk_rel"], v["blk_worst"]) for p, v in r.items()}, flush=True)
                    continue
                loss_ref = F.cross_entropy(logits_ref, y, reduction="sum") * igb
                loss_ref.backward()
                logits, loss, di, dt = eng.logits_head(fi, ft, y, igb, True)
                again = eng.logits_head(fi, ft, y, igb, True)
                torch.cuda.synchronize()
                r = {"logits": _metrics(logits, logits_ref.detach(), grid=(B,)),
                     "logits_cols": _metrics(logits.t(), logits_ref.detach().t(), grid=(Cn,)),
                     "loss": [float(loss), float(loss_ref)],
                     "d_img": _metrics(di, fid.grad, grid=(B,)), "d_txt": _metrics(dt, ftd.grad, grid=(Cn,)),
                     "repeat_bitwise": all(bool(torch.equal(a, b)) for a, b in zip((logits, loss, di, dt), again))}
                # label classes carry (p - 1) / 8B, the others p / 8B: each group per class at its own scale (BLK_FLOOR)
                lab = torch.zeros(Cn, dtype=torch.bool, device=dev)
                lab[y] = True
                if bool((~lab).any()):
                    r["d_txt_label"] = _metrics(dt[lab], ftd.grad[lab], grid=(int(lab.sum()),))
                    r["d_txt_other"] = _metrics(dt[~lab], ftd.grad[~lab], grid=(int((~lab).sum()),))
                if (B, Cn) == (32, 1000):
                    # class shard of one rank of eight: each class's logit is computed on its own
                    lo = 250
                    shard, _, _, _ = eng.logits_head(fi, ft[lo:lo + 125].contiguous(), None, igb, False)
                    torch.cuda.synchronize()
                    r["shard_bitwise"] = bool(torch.equal(shard, logits[:, lo:lo + 125]))
                # backward of the logits alone (module-level autograd path) at the same width
                dl = torch.randn(B, Cn, device=dev)
                fid.grad = None; ftd.grad = None
                (scale * F.normalize(fid, dim=-1) @ F.normalize(ftd, dim=-1).t()).backward(dl.double())
                di2, dt2 = eng.logits_backward(fi, ft, dl)
                torch.cuda.synchronize()
                r["bwd_img"] = _metrics(di2, fid.grad, grid=(B,))
                r["bwd_txt"] = _metrics(dt2, ftd.grad, grid=(Cn,))
                res[key] = r
                print(key, {p: (v["blk_rel"], v["blk_worst"]) for p, v in r.items() if isinstance(v, dict)},
                      r["loss"], r["repeat_bitwise"], r.get("shard_bitwise"), flush=True)
        del eng
    _feature_heads(res, dev)
    _feature_heads(res, dev, "ViT-L/14")


def _feature_heads(res, dev, arch_name="ViT-B/16"):
    """Feature heads (gather_ln_kernel + split-K sgemm, csrc/head.cu) at the widths of `arch_name` (ViT-B/16: vision
    768 -> 512, text 512 -> 512; ViT-L/14: vision 1024 -> 768, text 768 -> 768) on a one-layer-per-tower handle without
    pruning, so that x_in[layers] holds every row of the tower output: f_img = LN_post(x[:, 0]) @ proj and
    f_txt = ln_final(x[c, eot_c]) @ text_projection against fp64, per sequence."""
    import dataclasses
    import torch
    import torch.nn.functional as F
    from mudpt_b200 import _lib, synthetic as syn
    from mudpt_b200.engine import Engine
    arch = dataclasses.replace(syn.ARCHS[arch_name], vision_layers=1, transformer_layers=1)
    tag = "" if arch_name == "ViT-B/16" else "_" + arch_name.replace("/", "").replace("-", "").lower()
    sd = syn.synthetic_clip_state_dict(arch, 0)
    ad = dict(zip(["embed_dim", "image_resolution", "vision_layers", "vision_width", "vision_patch_size", "context_length",
                   "vocab_size", "transformer_width", "transformer_heads", "transformer_layers"], arch.astuple()))
    eng = Engine(ad, 2, 1, dev)
    eng.load_clip_weights(sd)
    _lib.check(eng.lib.mudpt_set_option(eng.h, b"prune", 0), eng.h)
    g = torch.Generator().manual_seed(4)
    dv, dt = arch.vision_width, arch.transformer_width
    eps = 1e-5
    # vision: the CLS row of each image
    B = 5
    img = syn.synthetic_images(B, arch.image_resolution, seed=4).to(dev)
    f_img = eng.vision_forward(img, (0.1 * torch.randn(1, 2, dv, generator=g)).to(dev))
    torch.cuda.synchronize()
    x = eng.debug_buffer(0, "x_in", 1, torch.float32).view(B, -1, dv)
    ref = F.layer_norm(x[:, 0].double(), (dv,), sd["visual.ln_post.weight"].double().to(dev),
                       sd["visual.ln_post.bias"].double().to(dev), eps) @ sd["visual.proj"].double().to(dev)
    res["feature_head_image" + tag] = _metrics(f_img, ref, grid=(B,))
    # text: the EOT row of each class, at different positions (and one at the last of the truncated length)
    eot = torch.tensor([3, 9, 4, 20, 7, 12, 5, 20, 16], dtype=torch.int64)
    Cn, seq_len = eot.numel(), int(eot.max()) + 1
    emb = torch.randn(Cn, arch.context_length, dt, generator=g) * 0.02
    eng.text_set_classes(emb, eot, seq_len)
    f_txt = eng.text_forward((0.02 * torch.randn(1, 2, dt, generator=g)).to(dev), True)
    torch.cuda.synchronize()
    x = eng.debug_buffer(1, "x_in", 1, torch.float32).view(Cn, seq_len, dt)
    xe = x[torch.arange(Cn, device=dev), eot.to(dev)]
    ref = F.layer_norm(xe.double(), (dt,), sd["ln_final.weight"].double().to(dev), sd["ln_final.bias"].double().to(dev),
                       eps) @ sd["text_projection"].double().to(dev)
    res["feature_head_text" + tag] = _metrics(f_txt, ref, grid=(Cn,))
    print("feature heads", arch_name, res["feature_head_image" + tag], res["feature_head_text" + tag], flush=True)
    del eng


def group_model_tiny(res):
    for name in ["tiny_a", "tiny_b", "tiny_c", "tiny_d"]:
        _compare_model(name, res)


def group_model_vitb16(res):
    _compare_model("vitb16_cfg1", res)


def run_group(name):
    res = {}
    t0 = time.time()
    try:
        globals()["group_" + name](res)
        res["_status"] = "ok"
    except Exception:
        res["_status"] = "exception"
        res["_trace"] = traceback.format_exc()
        print(res["_trace"], flush=True)
    res["_seconds"] = time.time() - t0
    return res


def main():
    args = sys.argv[1:]
    if args and args[0] == "--child":
        name = args[1]
        res = run_group(name)
        with open(args[2], "w") as f:
            json.dump(res, f, indent=1)
        return
    groups = args or GROUPS
    outdir = os.path.join(ROOT, "gpurun_out")
    os.makedirs(outdir, exist_ok=True)
    tag = os.environ.get("MUDPT_BRINGUP_TAG", "prod")
    allres = {}
    for gname in groups:
        path = os.path.join(outdir, f"bringup_{tag}_{gname}.json")
        print(f"===== group {gname} ({tag}) =====", flush=True)
        try:
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", gname, path], timeout=420)
            rc = p.returncode
        except subprocess.TimeoutExpired:
            rc = "timeout"
        if os.path.exists(path):
            allres[gname] = json.load(open(path))
        else:
            allres[gname] = {"_status": f"died rc={rc}"}
        print(f"===== group {gname}: {allres[gname].get('_status')} rc={rc} =====", flush=True)
    with open(os.path.join(outdir, f"bringup_{tag}.json"), "w") as f:
        json.dump(allres, f, indent=1)


if __name__ == "__main__":
    main()

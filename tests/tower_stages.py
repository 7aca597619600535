"""Stage-by-stage parity of a transformer tower, teacher-forced from the tower's own saved operands.

Every stage of every block is compared with fp64 computed from the operands the tower itself stored for that stage: the
residual rows x_in[i] / x_mid[i] (fp32), qkv[i], o[i] and the c_fc pre-activation h[i] (bf16), the log2-domain
log-sum-exp lse[i].  Each comparison therefore holds exactly one kernel's rounding, and the unit-test bounds of
tests/test_gpu_parity.py apply block by block unchanged:

  stage      reference (fp64)                                   block                    bound
  splice     prompt rows of x_in[i] = prompts[i]                sequence                 bitwise
  ln1_qkv    LN1(x_in[i]) W_in^T + b_in  vs qkv[i]               128 x 128 tile           BF16_REL; fused LayerNorm:
  ln2_fc     LN2(x_mid[i]) W_fc^T + b_fc vs h[i]                 128 x 128 tile           max(1.6 x unfused emulation, 6e-3)
  attn       softmax(q k^T / 8) v  vs o[i]                       (sequence, head)         BF16_REL
  lse        log2 sum exp(q k^T / 8)  vs lse[i]                  (sequence, head)         LSE2_REF_ABS, every query row
  out_proj   update x_mid[i] - x_in[i]  vs o[i] W_out^T + b_out  128 x 128 tile           BF16_REL
  c_proj     update x_in[i+1] - x_mid[i]  vs QuickGELU(h[i]) W_pr^T + b_pr   tile          BF16_REL
  last_block the pruned last block on the CLS / EOT rows, then the feature head, vs the features     sequence  BF16_REL
  head       LN(x_in[layers][sel]) proj  vs the features         sequence                 F32_REL

The updates, not the residual stream, are compared in out_proj / c_proj: the stream's magnitude would dilute an error of
the update (a bias lost on one tile).  The prompt rows that the next block's splice overwrites are left out of c_proj;
the splice stage checks them.  "Fused" is the rule of the fused-LayerNorm GEMM modes 7 / 8 (test_gpu_parity): the folded
form's error on a tile is held to 1.6 x the error of the stand-alone form (bf16(LN(x)) @ bf16(W), fp32 sums) on the same
tile, with a floor of 6e-3.

Used by tests/test_tower_parity.py (the native towers) and tests/test_tower_parity_host.py (an fp64 CPU tower with
injected faults, which these checks must find and name)."""
from __future__ import annotations

from dataclasses import dataclass
from typing import Callable, Dict, List, Optional, Sequence

import torch
import torch.nn.functional as F

from tests.gpu_bringup import GEMM_TILE, _attn_blocks, _attn_lse2_ref, _attn_ref, _block_rel
from tests.test_gpu_parity import BF16_REL, F32_REL, LSE2_REF_ABS

LN_EPS = 1e-5
FUSED_LN_FLOOR = 6e-3
STAGES = ("stem", "splice", "ln1_qkv", "attn", "lse", "out_proj", "ln2_fc", "c_proj", "last_block", "head", "d_prompts",
          "d_x0", "d_images")
BLOCK_KEYS = ("ln_1.weight", "ln_1.bias", "attn.in_proj_weight", "attn.in_proj_bias", "attn.out_proj.weight",
              "attn.out_proj.bias", "ln_2.weight", "ln_2.bias", "mlp.c_fc.weight", "mlp.c_fc.bias", "mlp.c_proj.weight",
              "mlp.c_proj.bias")


@dataclass
class Geometry:
    """Row layout of a tower: sequence s holds rows [off[s], off[s] + lengths[s]) (padded towers: equal lengths)."""
    lengths: List[int]
    H: int
    causal: bool
    row0: int               # position of the first prompt token in a sequence
    n_ctx: int
    spliced: Sequence[int]  # layers whose input carries that layer's deep prompt rows
    sel: List[int]          # absolute row per sequence that the feature head reads (CLS / EOT)

    @property
    def off(self) -> List[int]:
        o = [0]
        for n in self.lengths:
            o.append(o[-1] + n)
        return o

    @property
    def S(self) -> int:
        return len(self.lengths)

    def prompt_rows(self, device) -> torch.Tensor:
        """[S, n_ctx] absolute rows of the prompt tokens."""
        off = torch.tensor(self.off[:-1], device=device)
        return off[:, None] + self.row0 + torch.arange(self.n_ctx, device=device)[None]


class Report:
    """Worst block ratio (error / bound) per (layer, stage) and where it occurs."""

    def __init__(self):
        self.rows = []  # (layer, stage, ratio, block)

    def add(self, layer: int, stage: str, ratio: float, block):
        self.rows.append((layer, stage, float(ratio), tuple(block)))

    def worst(self) -> Dict[str, tuple]:
        """stage -> (ratio, layer, block) of its worst block over all layers"""
        out = {}
        for layer, stage, r, blk in self.rows:
            if stage not in out or not r <= out[stage][0]:
                out[stage] = (r, layer, blk)
        return {s: out[s] for s in STAGES if s in out}

    def failures(self) -> List[tuple]:
        """(layer, stage, ratio, block) over bound (NaN included), in the tower's order: layer, then stage"""
        bad = [r for r in self.rows if not r[2] <= 1.0]
        return sorted(bad, key=lambda r: (r[0], STAGES.index(r[1])))

    def table(self, title: str) -> str:
        lines = [f"{title}: worst block ratio (error / bound) per stage"]
        for s, (r, layer, blk) in self.worst().items():
            lines.append(f"  {s:<10} {r:9.3g}  layer {layer:<3} block {list(blk)}")
        return "\n".join(lines)


def _worst(ratio: torch.Tensor, names: Callable[[int], tuple]):
    ratio = torch.where(torch.isnan(ratio), torch.full_like(ratio, float("inf")), ratio).flatten()
    i = int(ratio.argmax())
    return float(ratio[i]), names(i)


def gemm_tiles(out: torch.Tensor, ref: torch.Tensor, emul: Optional[torch.Tensor] = None):
    """(worst ratio, (row, column) of its tile) of `out` against `ref` per 128 x 128 tile: bound BF16_REL, or with the
    stand-alone emulation `emul` the fused-LayerNorm rule max(1.6 x emul's error on the tile, 6e-3)."""
    blk = _block_rel(out, ref, tile=GEMM_TILE)
    bound = torch.full_like(blk, BF16_REL) if emul is None else (1.6 * _block_rel(emul, ref, tile=GEMM_TILE)).clamp_min(FUSED_LN_FLOOR)
    cols = -(-ref.shape[1] // GEMM_TILE[1])
    return _worst(blk / bound, lambda i: ((i // cols) * GEMM_TILE[0], (i % cols) * GEMM_TILE[1]))


def per_row(out: torch.Tensor, ref: torch.Tensor, bound: float, names: Optional[Callable[[int], tuple]] = None):
    blk = _block_rel(out, ref, grid=(out.shape[0],))
    return _worst(blk / bound, names or (lambda i: (i,)))


def ln_gemm_stage(x, g, b, W, bias, out, fused: bool):
    """LayerNorm + Linear: `out` (bf16, the tower's) against fp64 LN(x) W^T + bias from the tower's fp32 rows x."""
    d = x.shape[1]
    ref = F.layer_norm(x.double(), (d,), g.double(), b.double(), LN_EPS) @ W.double().t() + bias.double()
    emul = None
    if fused:
        a = F.layer_norm(x.float(), (d,), g.float(), b.float(), LN_EPS).bfloat16().float()
        emul = (a @ W.float().bfloat16().float().t() + bias.float()).bfloat16()
    return gemm_tiles(out, ref, emul)


def attention_stage(qkv: torch.Tensor, o: torch.Tensor, lse: torch.Tensor, geo: Geometry):
    """((ratio, (sequence, head)) of o, (ratio, (sequence, head)) of lse): o against fp64 attention per (sequence, head) at
    BF16_REL, lse (flat; sequence s holds [H, len_s] at off[s] * H) at LSE2_REF_ABS on every query row.  Sequences of
    equal length are checked together."""
    H, dev = geo.H, qkv.device
    off = geo.off
    best_o, best_l = (-1.0, None), (-1.0, None)
    for n in sorted(set(geo.lengths)):
        seqs = [s for s, ln in enumerate(geo.lengths) if ln == n]
        base = torch.tensor([off[s] for s in seqs], device=dev)
        rows = (base[:, None] + torch.arange(n, device=dev)[None]).flatten()
        q = qkv[rows].double()
        ref = _attn_ref(q, len(seqs), n, H, geo.causal)
        ro = _block_rel(_attn_blocks(o[rows], len(seqs), n, H), _attn_blocks(ref, len(seqs), n, H), grid=(len(seqs), H)) / BF16_REL
        li = (base[:, None] * H + torch.arange(H * n, device=dev)[None]).flatten()
        lerr = (lse[li].double().view(len(seqs), H, n) - _attn_lse2_ref(q, len(seqs), n, H, geo.causal)).abs().amax(-1)
        name = lambda i: (seqs[i // H], i % H)  # noqa: E731
        wo, wl = _worst(ro, name), _worst(lerr / LSE2_REF_ABS, name)
        best_o = best_o if wo[0] <= best_o[0] else wo
        best_l = best_l if wl[0] <= best_l[0] else wl
    return best_o, best_l


def quick_gelu(x):
    return x * torch.sigmoid(1.702 * x)


def check_layer(rep: Report, i: int, ops: Callable[[str, int], torch.Tensor], w: Dict[str, torch.Tensor], geo: Geometry,
                prompts: Optional[torch.Tensor], fused: bool, last_pruned: bool):
    """Every stage of block i.  ops(name, layer) returns the tower's saved buffer as [rows, width] (lse: flat);
    w: the block's weights under BLOCK_KEYS; prompts [depth, n_ctx, d] (fp32, as the tower got them)."""
    x = ops("x_in", i)
    if i in geo.spliced:
        pr = geo.prompt_rows(x.device)
        same = (x[pr].view(torch.int32) == prompts[i].to(x.device).view(torch.int32)[None]).all(-1).all(-1)  # [S]
        bad = (~same).nonzero()
        rep.add(i, "splice", 0.0 if bad.numel() == 0 else float("inf"), (int(bad[0]) if bad.numel() else 0,))
    qkv = ops("qkv", i)
    rep.add(i, "ln1_qkv", *ln_gemm_stage(x, w["ln_1.weight"], w["ln_1.bias"], w["attn.in_proj_weight"], w["attn.in_proj_bias"], qkv, fused))
    o = ops("o", i)
    ra, rl = attention_stage(qkv, o, ops("lse", i), geo)
    rep.add(i, "attn", *ra)
    rep.add(i, "lse", *rl)
    if last_pruned:
        return
    xm = ops("x_mid", i)
    ref = o.double() @ w["attn.out_proj.weight"].double().t() + w["attn.out_proj.bias"].double()
    rep.add(i, "out_proj", *gemm_tiles(xm.double() - x.double(), ref))
    h = ops("h", i)
    rep.add(i, "ln2_fc", *ln_gemm_stage(xm, w["ln_2.weight"], w["ln_2.bias"], w["mlp.c_fc.weight"], w["mlp.c_fc.bias"], h, fused))
    ref = quick_gelu(h.double()) @ w["mlp.c_proj.weight"].double().t() + w["mlp.c_proj.bias"].double()
    upd = ops("x_in", i + 1).double() - xm.double()
    if i + 1 in geo.spliced:
        pr = geo.prompt_rows(upd.device).flatten()
        upd[pr] = ref[pr]
    rep.add(i, "c_proj", *gemm_tiles(upd, ref))


def _ln(x, g, b):
    return F.layer_norm(x, (x.shape[-1],), g.double(), b.double(), LN_EPS)


def last_block_features(x: torch.Tensor, qkv: torch.Tensor, w: Dict[str, torch.Tensor], geo: Geometry, ln_g, ln_b, proj):
    """fp64 features of the last block evaluated on the selected rows only (what the pruned tower computes): attention of
    the selected query over every visible key of its sequence, out-proj + residual, MLP + residual, then LN and proj."""
    dev, H = qkv.device, geo.H
    d = x.shape[1]
    off, Lm = geo.off, max(geo.lengths)
    sel = torch.tensor(geo.sel, device=dev)
    start = torch.tensor(off[:-1], device=dev)
    n = torch.tensor(geo.lengths, device=dev)
    j = torch.arange(Lm, device=dev)[None]
    keys = (start[:, None] + j).clamp_max(qkv.shape[0] - 1)        # [S, Lm]
    vis = j < n[:, None]
    if geo.causal:
        vis = vis & (j <= (sel - start)[:, None])
    q = qkv[sel, :d].double().view(-1, H, 1, 64)
    kv = qkv[keys].double()
    k = kv[..., d:2 * d].reshape(-1, Lm, H, 64).permute(0, 2, 3, 1)
    v = kv[..., 2 * d:].reshape(-1, Lm, H, 64).permute(0, 2, 1, 3)
    s = (q @ k) * 0.125 + torch.where(vis, 0.0, float("-inf")).to(torch.float64)[:, None, None]
    att = (torch.softmax(s, -1) @ v).reshape(-1, d)
    xm = x[sel].double() + att @ w["attn.out_proj.weight"].double().t() + w["attn.out_proj.bias"].double()
    hh = _ln(xm, w["ln_2.weight"], w["ln_2.bias"]) @ w["mlp.c_fc.weight"].double().t() + w["mlp.c_fc.bias"].double()
    xo = xm + quick_gelu(hh) @ w["mlp.c_proj.weight"].double().t() + w["mlp.c_proj.bias"].double()
    return _ln(xo, ln_g, ln_b) @ proj.double()


def check_tower(ops, weights: Callable[[int], Dict[str, torch.Tensor]], layers: int, geo: Geometry, prompts, fused: bool,
                pruned: bool, features: torch.Tensor, ln_g, ln_b, proj, rep: Optional[Report] = None) -> Report:
    """Every block and the feature head of a tower after one forward; `features` are the tower's output [S, e], ln_g /
    ln_b / proj its final LayerNorm and projection."""
    rep = rep or Report()
    for i in range(layers):
        last_pruned = pruned and i == layers - 1
        check_layer(rep, i, ops, weights(i), geo, prompts, fused, last_pruned)
    if pruned:
        ref = last_block_features(ops("x_in", layers - 1), ops("qkv", layers - 1), weights(layers - 1), geo, ln_g, ln_b, proj)
        rep.add(layers - 1, "last_block", *per_row(features, ref, BF16_REL))
    else:
        ref = _ln(ops("x_in", layers)[torch.tensor(geo.sel, device=features.device)].double(), ln_g, ln_b) @ proj.double()
        rep.add(layers, "head", *per_row(features, ref, F32_REL))
    return rep


# ------------------------------------------------------------------------------------------------ backward
# The backward keeps no per-layer gradients, so it is checked end to end through short (3-layer) towers at the real widths
# and row counts: the tower's prompt (and input / image) gradients against fp64 autograd of the same blocks from the
# tower's own input x_in[0] and the same d_f.  Each block (a (layer, token) row of d_prompts, a row of d_x0, a patch-row
# band of an image) is held to max(BF16_REL, 1.6 x the error that an fp32 emulation with the native roundings makes on it),
# the rule of the attention and fused-LayerNorm tests.  The emulation (emulate=True below) rounds to bf16 where the native
# stand-alone backward does: the GEMM operands (LayerNorm outputs and their gradients, qkv / dqkv, o / do, h / dh, the
# QuickGELU output, the bf16 copy of the residual gradient that the dgrad GEMMs read, the weights), attention P and dS
# with D as in gpu_bringup._attn_emul_bf16, the residual gradient itself between the LayerNorm backward kernels when it
# travels in bf16 (grad_stream_bf16).  Fused-LayerNorm forwards are emulated as they compute: x_hat from the bf16 row and
# the exact statistics, gamma folded into the bf16 weight; the LayerNorm backwards that read that bf16 row form x_hat
# the same way.

class _Round(torch.autograd.Function):
    """bf16 rounding of the value (fwd) and / or of the gradient that flows back through it (bwd)"""

    @staticmethod
    def forward(ctx, x, fwd, bwd):
        ctx.bwd = bwd
        return x.bfloat16().to(x.dtype) if fwd else x.clone()

    @staticmethod
    def backward(ctx, g):
        return (g.bfloat16().to(g.dtype) if ctx.bwd else g), None, None


class _EmulAttention(torch.autograd.Function):
    """Attention of S sequences of L tokens as the kernels compute it (gpu_bringup._attn_emul_bf16), forward and backward"""

    @staticmethod
    def forward(ctx, qkv, S, L, H, causal):
        from tests.gpu_bringup import _attn_emul_bf16
        ctx.save_for_backward(qkv)
        ctx.shape = (S, L, H, causal)
        o, _, _, _ = _attn_emul_bf16(qkv, torch.zeros(S * L, H * 64, device=qkv.device), S, L, H, causal)
        return o.to(qkv.dtype)

    @staticmethod
    def backward(ctx, do):
        from tests.gpu_bringup import _attn_emul_bf16
        qkv, = ctx.saved_tensors
        _, dq, dk, dv = _attn_emul_bf16(qkv, do, *ctx.shape)
        return torch.cat([dq, dk, dv], 1).to(qkv.dtype), None, None, None, None


class _LayerNormX16(torch.autograd.Function):
    """x_hat of the fused-LayerNorm formulation: (bf16(x) - mean) rstd with the exact row statistics, forward (the GEMM
    reads the bf16 row and applies the statistics in its epilogue) and backward (the LayerNorm backward kernels read the
    same bf16 row)"""

    @staticmethod
    def forward(ctx, x):
        mean = x.mean(1, keepdim=True)
        rstd = torch.rsqrt(x.var(1, unbiased=False, keepdim=True) + LN_EPS)
        ctx.save_for_backward(x, mean, rstd)
        return (x.bfloat16().to(x.dtype) - mean) * rstd

    @staticmethod
    def backward(ctx, g):
        x, mean, rstd = ctx.saved_tensors
        xh = (x.bfloat16().to(x.dtype) - mean) * rstd
        return rstd * (g - g.mean(1, keepdim=True) - xh * (g * xh).mean(1, keepdim=True))


def _attention(qkv, geo: Geometry, emulate: bool):
    """Attention over the tower's row layout, differentiable; sequences of equal length run together."""
    H, d = geo.H, qkv.shape[1] // 3
    off = geo.off
    out = torch.zeros(qkv.shape[0], d, device=qkv.device, dtype=qkv.dtype)
    for n in sorted(set(geo.lengths)):
        seqs = [s for s, ln in enumerate(geo.lengths) if ln == n]
        base = torch.tensor([off[s] for s in seqs], device=qkv.device)
        rows = (base[:, None] + torch.arange(n, device=qkv.device)[None]).flatten()
        q = qkv[rows]
        o = _EmulAttention.apply(q, len(seqs), n, H, geo.causal) if emulate else _attn_ref(q, len(seqs), n, H, geo.causal)
        out = out.index_put((rows,), o)
    return out


def tower_grads(x0, prompts, weights: Callable[[int], Dict[str, torch.Tensor]], layers: int, geo: Geometry, ln_g, ln_b, proj,
                d_f, emulate: bool, grad_stream_bf16: bool, ln_x16=frozenset()):
    """Runs the tower from its input rows x0 [rows, d] (the prompt rows of the spliced layers are replaced by prompts[i],
    which must require grad), the feature head on geo.sel, and back-propagates d_f.  fp64 without rounding, or with
    emulate=True fp32 with the native roundings; ln_x16 holds the (layer, 1 | 2) LayerNorms of the fused formulation
    (_LayerNormX16, gamma folded into the bf16 weight, no bf16 LayerNorm output).  x0 may be a leaf or come from a differentiable stem."""
    dt = torch.float32 if emulate else torch.float64

    def R(t, fwd=True, bwd=True):
        return _Round.apply(t, fwd, bwd) if emulate else t

    def lin(a, W, b):
        return a @ (W.bfloat16() if emulate else W).to(dt).t() + b.to(dt)

    def ln(t, g, b):
        return F.layer_norm(t, (t.shape[1],), g.to(dt), b.to(dt), LN_EPS)

    def ln_lin(t, g, b, W, bias, key):
        """LayerNorm -> Linear; in the emulation the stand-alone form bf16(LN(x)) @ bf16(W) or the fused one
        x_hat16 @ bf16(W gamma) + (bias + W beta)"""
        if not emulate:
            return lin(ln(t, g, b), W, bias)
        if key in ln_x16:
            return lin(R(_LayerNormX16.apply(t), False, True), W * g[None], bias + W @ b)
        return lin(R(ln(t, g, b)), W, bias)

    x = x0.to(dt)
    pr = geo.prompt_rows(x.device).flatten() if geo.n_ctx else None
    for i in range(layers):
        w = weights(i)
        if i in geo.spliced:
            x = x.index_put((pr,), prompts[i].to(dt).repeat(geo.S, 1))
        qkv = R(ln_lin(x, w["ln_1.weight"], w["ln_1.bias"], w["attn.in_proj_weight"], w["attn.in_proj_bias"], (i, 1)))
        o = R(_attention(qkv, geo, emulate))
        x = R(x + R(lin(o, w["attn.out_proj.weight"], w["attn.out_proj.bias"]), False), False, grad_stream_bf16)
        h = R(ln_lin(x, w["ln_2.weight"], w["ln_2.bias"], w["mlp.c_fc.weight"], w["mlp.c_fc.bias"], (i, 2)))
        g = R(quick_gelu(h), True, False)
        x = R(x + R(lin(g, w["mlp.c_proj.weight"], w["mlp.c_proj.bias"]), False), False, grad_stream_bf16)
    f = ln(x[torch.tensor(geo.sel, device=x.device)], ln_g, ln_b) @ proj.to(dt)
    f.backward(d_f.to(dt))


def grad_blocks(got, ref, emul, grid, names: Callable[[int], tuple]):
    """(worst ratio, block) of the tower's gradient `got` against the fp64 `ref`, per block of `grid`, each bounded by
    max(BF16_REL, 1.6 x the emulation's error on that block)"""
    bound = (1.6 * _block_rel(emul, ref, grid=grid)).clamp_min(BF16_REL)
    return _worst(_block_rel(got, ref, grid=grid) / bound, names)

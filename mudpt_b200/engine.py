"""Host-side owner of the native handle: pushes the frozen CLIP weights through the C ABI once and
exposes the tower / head calls as torch.autograd.Functions.

PyTorch is used for device memory, streams and autograd plumbing only; every FLOP of the towers
runs in libmudpt_b200.so (include/mudpt_b200.h).  No fallback: a missing library or GPU raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, List, Optional, Tuple

import torch

from . import _lib


def text_lengths(eot: torch.Tensor, mode, full_len: int, min_len: int) -> Tuple[int, Optional[List[int]]]:
    """Token counts the text tower runs for classes whose EOT tokens sit at positions `eot` [C].

    mode True: one length for all classes, max(eot) + 1; False: all `full_len` positions; "per_class": class c runs
    max(eot_c + 1, min_len) tokens (a ragged tower).  Every length is at least `min_len` (SOT + the n_ctx prompt rows).
    Dropping the tokens after EOT is exact under the causal mask.  Returns (padded length, per-class lengths or None)."""
    if mode == "per_class":
        lengths = [max(int(e) + 1, min_len) for e in eot.tolist()]
        return max(lengths), lengths
    if mode is not True and mode is not False:
        raise ValueError(f"mudpt_b200: text truncation mode must be True, False or 'per_class', not {mode!r}")
    seq_len = int(eot.max()) + 1 if mode else int(full_len)
    return max(seq_len, min_len), None


def packed_offsets(lengths: List[int]) -> List[int]:
    """Row offsets [C + 1] of the packed ragged layout: class c occupies rows [off[c], off[c + 1])."""
    off = [0]
    for n in lengths:
        off.append(off[-1] + int(n))
    return off


class Engine:
    """One native handle (one GPU).  Not thread-safe, like the handle itself."""

    def __init__(self, arch: Dict[str, int], n_ctx: int, depth: int, device: torch.device):
        if device.type != "cuda":
            raise RuntimeError("mudpt_b200: the hot path runs on a CUDA device only (no CPU fallback)")
        self.lib = _lib.load()
        self.device = device
        self.n_ctx, self.depth = int(n_ctx), int(depth)
        self.arch = dict(arch)
        cfg = _lib.Config(
            embed_dim=arch["embed_dim"], image_resolution=arch["image_resolution"],
            vision_layers=arch["vision_layers"], vision_width=arch["vision_width"],
            vision_patch_size=arch["vision_patch_size"], context_length=arch["context_length"],
            transformer_width=arch["transformer_width"], transformer_heads=arch["transformer_heads"],
            transformer_layers=arch["transformer_layers"], n_ctx=n_ctx, prompt_depth=depth,
            device=device.index if device.index is not None else torch.cuda.current_device())
        h = C.c_void_p()
        _lib.check(self.lib.mudpt_create(C.byref(cfg), C.byref(h)))
        self.h = h
        self.vision_gen = 0  # generation counters: a backward must match the latest forward
        self.vision_batch = 0  # images of the latest vision_forward
        self.text_gen = 0
        self.n_classes = 0
        self.text_len = 0
        self.class_key = None  # identifies the class set currently resident in the text tower
        self._side = None

    def side_stream(self) -> torch.cuda.Stream:
        """Second stream of this engine's device (the two towers use disjoint workspaces of the handle)."""
        if self._side is None:
            # MUDPT_SIDE_PRIORITY: CUDA stream priority of the vision stream (-1 = high).  Measured: ANY priority difference
            # between the two towers' streams is slower (per-rank shapes 6.3 -> 7.2 ms, either way round): equal priorities
            prio = int(os.environ.get("MUDPT_SIDE_PRIORITY", "0"))
            self._side = torch.cuda.Stream(self.device, priority=prio)
        return self._side

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.lib.mudpt_destroy(self.h)
                self.h = None
        except Exception:
            pass

    # ---------------------------------------------------------------- weights
    def load_clip_weights(self, state_dict: Dict[str, torch.Tensor]) -> None:
        """`state_dict` uses the reference CLIP.state_dict() names (clip/model.py:667-779)."""
        st = _lib.stream_ptr(self.device)
        keep = []
        for name, t in state_dict.items():
            if name.startswith("token_embedding") or "visual_ctx" in name:
                continue  # not part of the frozen towers
            w = t.detach().to(device=self.device, dtype=torch.float32).contiguous()
            keep.append(w)
            rc = self.lib.mudpt_set_weight(self.h, name.encode(), w.data_ptr(), w.numel(), st)
            _lib.check(rc, self.h)
        torch.cuda.current_stream(self.device).synchronize()  # staging copies may now be freed
        _lib.check(self.lib.mudpt_weights_complete(self.h), self.h)

    # ---------------------------------------------------------------- raw calls
    def _check_f32(self, t: torch.Tensor, shape=None):
        if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
            raise RuntimeError("mudpt_b200: expected a contiguous fp32 CUDA tensor")
        if shape is not None and tuple(t.shape) != tuple(shape):
            raise RuntimeError(f"mudpt_b200: expected shape {tuple(shape)}, got {tuple(t.shape)}")

    def _vision(self, fn, images: torch.Tensor, prompts: torch.Tensor) -> torch.Tensor:
        a = self.arch
        R = a["image_resolution"]
        images = images.to(torch.float32).contiguous()
        self._check_f32(images, (images.shape[0], 3, R, R))
        prompts = prompts.contiguous()
        self._check_f32(prompts, (self.depth, self.n_ctx, a["vision_width"]))
        out = torch.empty(images.shape[0], a["embed_dim"], device=self.device, dtype=torch.float32)
        _lib.check(fn(self.h, images.data_ptr(), images.shape[0], prompts.data_ptr(), out.data_ptr(), _lib.stream_ptr(self.device)),
                   self.h)
        return out

    def vision_forward(self, images: torch.Tensor, prompts: torch.Tensor) -> torch.Tensor:
        out = self._vision(self.lib.mudpt_vision_forward, images, prompts)
        self.vision_gen += 1
        self.vision_batch = out.shape[0]
        return out

    def vision_infer(self, images: torch.Tensor, prompts: torch.Tensor) -> torch.Tensor:
        """vision_forward's result, bitwise, from the forward-only walk: no backward state is kept or touched (a pending
        vision_backward still differentiates the last vision_forward)."""
        return self._vision(self.lib.mudpt_vision_infer, images, prompts)

    def vision_backward(self, d_f_img: torch.Tensor) -> torch.Tensor:
        d_f_img = d_f_img.contiguous()
        self._check_f32(d_f_img)
        dP = torch.empty(self.depth, self.n_ctx, self.arch["vision_width"], device=self.device, dtype=torch.float32)
        _lib.check(self.lib.mudpt_vision_backward(self.h, d_f_img.data_ptr(), dP.data_ptr(),
                                                  _lib.stream_ptr(self.device)), self.h)
        return dP

    def vision_backward_images(self, d_f_img: torch.Tensor, want_prompts: bool = True):
        """(d_prompts or None, d_images [B, 3, R, R]) of the last vision_forward: the gradient w.r.t. the images as they
        were passed in, and (want_prompts) w.r.t. the prompt stack, as vision_backward."""
        d_f_img = d_f_img.contiguous()
        B, R = self.vision_batch, self.arch["image_resolution"]
        self._check_f32(d_f_img, (B, self.arch["embed_dim"]))
        d_img = torch.empty(B, 3, R, R, device=self.device, dtype=torch.float32)
        dP = None
        if want_prompts:
            dP = torch.empty(self.depth, self.n_ctx, self.arch["vision_width"], device=self.device, dtype=torch.float32)
        _lib.check(self.lib.mudpt_vision_backward_images(self.h, d_f_img.data_ptr(), dP.data_ptr() if dP is not None else None,
                                                         d_img.data_ptr(), _lib.stream_ptr(self.device)), self.h)
        return dP, d_img

    def vision_pgd_step(self, d_f_img: torch.Tensor, x_adv: torch.Tensor, x_clean: torch.Tensor, x_norm: torch.Tensor,
                        mean, std, eps: float, alpha: float) -> None:
        """One l-inf PGD step on the images of the last vision_forward, which were x_norm = (x_adv - mean) / std:
        x_adv <- clamp(clamp(x_adv + alpha * sign(dL/d x_adv), x_clean - eps, x_clean + eps), 0, 1) in place, and x_norm
        <- (x_adv - mean) / std, bitwise that PyTorch loop (include/mudpt_b200.h, mudpt_vision_pgd_step).  x_adv, x_clean,
        x_norm [B, 3, R, R] fp32 (x_norm may be the tensor the forward read); mean, std: 3 per-channel values."""
        d_f_img = d_f_img.contiguous()
        B, R = self.vision_batch, self.arch["image_resolution"]
        self._check_f32(d_f_img, (B, self.arch["embed_dim"]))
        for x in (x_adv, x_clean, x_norm):
            self._check_f32(x, (B, 3, R, R))
        mean_h, std_h = (_channels(v) for v in (mean, std))
        _lib.check(self.lib.mudpt_vision_pgd_step(self.h, d_f_img.data_ptr(), x_adv.data_ptr(), x_clean.data_ptr(),
                                                  x_norm.data_ptr(), mean_h, std_h, float(eps), float(alpha),
                                                  _lib.stream_ptr(self.device)), self.h)

    def text_set_classes(self, embeddings: torch.Tensor, eot: torch.Tensor, seq_len: int,
                         lengths: Optional[List[int]] = None) -> None:
        """embeddings [C, src_len, width] fp32; eot [C] int (position of the EOT token).  With `lengths` [C] the tower is
        ragged: class c runs its first lengths[c] tokens (packed rows, see text_lengths) and seq_len is ignored."""
        embeddings = embeddings.to(device=self.device, dtype=torch.float32).contiguous()
        Cn, src_len, _ = embeddings.shape
        eot_host = (C.c_int32 * Cn)(*[int(v) for v in eot.tolist()])
        if lengths is None:
            _lib.check(self.lib.mudpt_text_set_classes(self.h, embeddings.data_ptr(), Cn, src_len, int(seq_len), eot_host,
                                                       _lib.stream_ptr(self.device)), self.h)
        else:
            if len(lengths) != Cn:
                raise ValueError(f"mudpt_b200: {len(lengths)} lengths for {Cn} classes")
            len_host = (C.c_int32 * Cn)(*[int(v) for v in lengths])
            _lib.check(self.lib.mudpt_text_set_classes_ragged(self.h, embeddings.data_ptr(), Cn, src_len, len_host, eot_host,
                                                              _lib.stream_ptr(self.device)), self.h)
            seq_len = max(int(v) for v in lengths)
        torch.cuda.current_stream(self.device).synchronize()
        self.n_classes, self.text_len = Cn, int(seq_len)
        self.class_key = None

    def _text(self, fn, prompts: torch.Tensor, splice_layer0: bool, out: Optional[torch.Tensor]) -> torch.Tensor:
        prompts = prompts.contiguous()
        self._check_f32(prompts, (self.depth, self.n_ctx, self.arch["transformer_width"]))
        if out is None:
            out = torch.empty(self.n_classes, self.arch["embed_dim"], device=self.device, dtype=torch.float32)
        else:  # caller-owned destination (e.g. a peer-mapped buffer of the head's exchange)
            self._check_f32(out, (self.n_classes, self.arch["embed_dim"]))
        _lib.check(fn(self.h, prompts.data_ptr(), 1 if splice_layer0 else 0, out.data_ptr(), _lib.stream_ptr(self.device)), self.h)
        return out

    def text_forward(self, prompts: torch.Tensor, splice_layer0: bool = True, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        out = self._text(self.lib.mudpt_text_forward, prompts, splice_layer0, out)
        self.text_gen += 1
        return out

    def text_infer(self, prompts: torch.Tensor, splice_layer0: bool = True, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """text_forward's result, bitwise, from the forward-only walk (see vision_infer)."""
        return self._text(self.lib.mudpt_text_infer, prompts, splice_layer0, out)

    WORKSPACE_KINDS = {"train": 0, "infer": 1, "input": 2}

    def workspace_bytes(self, tower: str, kind: str) -> int:
        """Device bytes the handle holds for tower "vision" / "text": kind "train" (training workspace), "infer" (inference
        workspace) or "input" (the tower input: class set or stem output)."""
        b = C.c_int64()
        t = {"vision": 0, "text": 1}[tower]
        _lib.check(self.lib.mudpt_workspace_bytes(self.h, t, self.WORKSPACE_KINDS[kind], C.byref(b)), self.h)
        return int(b.value)

    def text_backward(self, d_f_txt: torch.Tensor, want_dx0: bool = False):
        d_f_txt = d_f_txt.contiguous()
        self._check_f32(d_f_txt)
        dP = torch.empty(self.depth, self.n_ctx, self.arch["transformer_width"], device=self.device, dtype=torch.float32)
        dx0 = None
        if want_dx0:
            dx0 = torch.empty(self.n_classes, self.text_len, self.arch["transformer_width"], device=self.device,
                              dtype=torch.float32)
        _lib.check(self.lib.mudpt_text_backward(self.h, d_f_txt.data_ptr(), dP.data_ptr(),
                                                dx0.data_ptr() if dx0 is not None else None,
                                                _lib.stream_ptr(self.device)), self.h)
        return dP, dx0

    def logits_head(self, f_img, f_txt, labels: Optional[torch.Tensor], inv_global_batch: float, want_grads: bool,
                    d_t_out: Optional[torch.Tensor] = None, text_grad: bool = True):
        """(logits, loss, d_f_img, d_f_txt); with want_grads and text_grad=False the text-feature gradient is not computed
        (None)."""
        f_img, f_txt = f_img.contiguous(), f_txt.contiguous()
        B, Cn = f_img.shape[0], f_txt.shape[0]
        logits = torch.empty(B, Cn, device=self.device, dtype=torch.float32)
        loss = torch.zeros((), device=self.device, dtype=torch.float32)
        d_i = torch.empty_like(f_img) if want_grads else None
        d_t = None
        if want_grads and text_grad:
            if d_t_out is not None:  # caller-owned destination (peer-mapped buffer)
                self._check_f32(d_t_out, tuple(f_txt.shape))
                d_t = d_t_out
            else:
                d_t = torch.empty_like(f_txt)
        if labels is not None:
            labels = labels.to(device=self.device, dtype=torch.int64).contiguous()
        _lib.check(self.lib.mudpt_logits_head(
            self.h, f_img.data_ptr(), f_txt.data_ptr(), labels.data_ptr() if labels is not None else None, B, Cn,
            float(inv_global_batch), logits.data_ptr(), loss.data_ptr(),
            d_i.data_ptr() if d_i is not None else None, d_t.data_ptr() if d_t is not None else None,
            _lib.stream_ptr(self.device)), self.h)
        return logits, loss, d_i, d_t

    def logits_backward(self, f_img, f_txt, dlogits):
        f_img, f_txt, dlogits = f_img.contiguous(), f_txt.contiguous(), dlogits.contiguous()
        d_i, d_t = torch.empty_like(f_img), torch.empty_like(f_txt)
        _lib.check(self.lib.mudpt_logits_backward(self.h, f_img.data_ptr(), f_txt.data_ptr(), dlogits.data_ptr(),
                                                  f_img.shape[0], f_txt.shape[0], d_i.data_ptr(), d_t.data_ptr(),
                                                  _lib.stream_ptr(self.device)), self.h)
        return d_i, d_t

    PROFILE_CATEGORIES = ("gemm_other", "attn_fwd", "attn_bwd", "ln_fwd", "ln_bwd", "splice", "head", "stem", "gemm_qkv", "gemm_out",
                          "gemm_fc", "gemm_proj", "gemm_dproj", "gemm_dfc", "gemm_dout", "gemm_dqkv")

    def profile_begin(self) -> None:
        _lib.check(self.lib.mudpt_profile_begin(self.h), self.h)

    def profile_end(self, peak_tflops: float = 0.0, hbm_gbs: float = 0.0) -> dict:
        """Per kernel class: ms, launches, algorithmic FLOPs and bytes -- and, with the two peaks given, `bound_ms`: the
        sum over the launches of max(FLOPs / peak, bytes / hbm), the time at the bound that applies to each launch."""
        n = len(self.PROFILE_CATEGORIES) * 5
        buf = (C.c_double * n)()
        _lib.check(self.lib.mudpt_profile_end_bound(self.h, buf, n, float(peak_tflops), float(hbm_gbs)), self.h)
        out = {c: {"ms": buf[i * 5], "launches": int(buf[i * 5 + 1]), "flops": buf[i * 5 + 2], "bytes": buf[i * 5 + 3],
                   "bound_ms": buf[i * 5 + 4]} for i, c in enumerate(self.PROFILE_CATEGORIES)}
        # "gemm" = every launch of the tcgen05 GEMM kernel (the per-GEMM entries stay beside it)
        out["gemm"] = {k: sum(v[k] for c, v in out.items() if c.startswith("gemm_")) for k in ("ms", "launches", "flops", "bytes", "bound_ms")}
        return out

    def launch_count(self) -> int:
        return int(self.lib.mudpt_launch_count(self.h))

    def debug_buffer(self, tower: int, name: str, layer: int, dtype: torch.dtype) -> torch.Tensor:
        """Copy of an internal activation buffer (tests only)."""
        p, n = C.c_void_p(), C.c_int64()
        _lib.check(self.lib.mudpt_debug_buffer(self.h, tower, name.encode(), layer, C.byref(p), C.byref(n)), self.h)
        out = torch.empty(n.value, device=self.device, dtype=dtype)
        torch.cuda.current_stream(self.device).synchronize()
        # device-to-device copy through torch: view the raw pointer via __cuda_array_interface__
        src = _from_ptr(p.value, n.value, dtype, self.device)
        out.copy_(src)
        return out


def _channels(v):
    """3 per-channel values (a sequence or a tensor of 3 elements) as a host fp32 array"""
    vals = torch.as_tensor(v, dtype=torch.float32).detach().cpu().flatten().tolist()
    if len(vals) != 3:
        raise ValueError(f"mudpt_b200: expected 3 per-channel values, got {len(vals)}")
    return (C.c_float * 3)(*vals)


def _from_ptr(ptr: int, numel: int, dtype: torch.dtype, device: torch.device) -> torch.Tensor:
    """View raw device memory as a tensor (tests / debugging only)."""
    itemsize = torch.empty((), dtype=dtype).element_size()

    class _Holder:
        pass

    h = _Holder()
    h.__cuda_array_interface__ = {
        "shape": (numel,), "typestr": {2: "<u2", 4: "<f4"}[itemsize], "data": (ptr, False), "version": 2}
    t = torch.as_tensor(h, device=device)
    return t.view(dtype) if t.dtype != dtype else t


# ------------------------------------------------------------------------------------------------
# autograd plumbing
# ------------------------------------------------------------------------------------------------

PROMPT_NAMES = ("ctx", "deep", "We", "be", "Wd", "bd", "vctx", "vdeep", "Wv", "bv")


def prompt_algebra_forward(lib, eps, ln_g, ln_b, pos, train):
    """(P_v, P_t, saved) = the two prompt stacks of MuDPT as functions of its 10 trainable tensors `train` (in
    PROMPT_NAMES order) -- trainers/mudpt.py:117-130, 143, 175; clip/model.py:534-541 -- in 2 native launches
    (mudpt_prompt_forward).  `saved` is what prompt_algebra_backward needs."""
    t = [x.detach().contiguous() for x in train]
    ctx, deep, vctx = t[0], t[1], t[6]
    n, dt = ctx.shape
    dv = vctx.shape[1]
    depth = deep.shape[0] + 1
    dev = ctx.device
    a = _lib.PromptArgs()
    a.n, a.depth, a.dt, a.dv, a.eps = n, depth, dt, dv, float(eps)
    frozen = [ln_g.detach().float().contiguous(), ln_b.detach().float().contiguous(), pos.detach().float().contiguous()]
    for k, x in zip(PROMPT_NAMES, t):
        setattr(a, k, x.data_ptr())
    a.ln_g, a.ln_b, a.pos = (x.data_ptr() for x in frozen)
    P_v = torch.empty(depth, n, dv, device=dev, dtype=torch.float32)
    P_t = torch.empty(depth, n, dt, device=dev, dtype=torch.float32)
    ln_in = torch.empty(n, dv, device=dev, dtype=torch.float32)
    a.P_v, a.P_t, a.ln_in = P_v.data_ptr(), P_t.data_ptr(), ln_in.data_ptr()
    _lib.check(lib.mudpt_prompt_forward(C.byref(a), _lib.stream_ptr(dev)))
    return P_v, P_t, (t, frozen, ln_in, float(eps))


def prompt_algebra_backward(lib, saved, dP_v, dP_t, grads=None):
    """Gradients of the 10 trainable tensors from (dP_v, dP_t) in 2 native launches (mudpt_prompt_backward).  Every
    element of every gradient is written (no accumulation): `grads` may be the views of a flat all-reduce bucket."""
    t, frozen, ln_in, eps = saved
    ctx, deep, vctx = t[0], t[1], t[6]
    n, dt = ctx.shape
    dv = vctx.shape[1]
    dev = ctx.device
    a = _lib.PromptArgs()
    a.n, a.depth, a.dt, a.dv, a.eps = n, deep.shape[0] + 1, dt, dv, eps
    for k, x in zip(PROMPT_NAMES, t):
        setattr(a, k, x.data_ptr())
    a.ln_g, a.ln_b, a.pos = (x.data_ptr() for x in frozen)
    a.ln_in = ln_in.data_ptr()
    dP_v, dP_t = dP_v.float().contiguous(), dP_t.float().contiguous()
    a.dP_v, a.dP_t = dP_v.data_ptr(), dP_t.data_ptr()
    u = torch.empty(n, dv, device=dev, dtype=torch.float32)
    if grads is None:
        grads = [torch.empty_like(x, dtype=torch.float32) for x in t]
    for g, x in zip(grads, t):
        if g.shape != x.shape or g.dtype != torch.float32 or not g.is_contiguous() or g.device != x.device:
            raise ValueError("mudpt_b200: prompt gradient buffer does not match its parameter")
    a.u = u.data_ptr()
    for k, g in zip(PROMPT_NAMES, grads):
        setattr(a, "d_" + k, g.data_ptr())
    _lib.check(lib.mudpt_prompt_backward(C.byref(a), _lib.stream_ptr(dev)))
    return grads


class PromptAlgebraFn(torch.autograd.Function):
    """prompt_algebra_forward / _backward behind autograd: 2 + 2 native launches instead of ~48 framework ops at the
    very start and end of the step.  `frozen` = (ln_pre.weight, ln_pre.bias, positional_embedding[1:1+n])."""

    NAMES = PROMPT_NAMES

    @staticmethod
    def forward(ctx_, lib, eps, ln_g, ln_b, pos, *train):
        P_v, P_t, saved = prompt_algebra_forward(lib, eps, ln_g, ln_b, pos, train)
        ctx_.lib, ctx_.saved = lib, saved
        return P_v, P_t

    @staticmethod
    def backward(ctx_, dP_v, dP_t):
        grads = prompt_algebra_backward(ctx_.lib, ctx_.saved, dP_v, dP_t)
        return (None, None, None, None, None, *grads)


class VisionTowerFn(torch.autograd.Function):
    """f_img = vision_tower(images; prompts).  Gradient flows to `prompts` and, when they require it, to `images` (the
    tensor as passed in); every CLIP weight is frozen (trainers/mudpt.py:205-212)."""

    @staticmethod
    def forward(ctx, engine: Engine, images, prompts):
        out = engine.vision_forward(images, prompts.detach())
        ctx.engine, ctx.gen = engine, engine.vision_gen
        return out

    @staticmethod
    def backward(ctx, d_out):
        e = ctx.engine
        if ctx.gen != e.vision_gen:
            raise RuntimeError("mudpt_b200: vision backward does not match the latest forward (activations were overwritten)")
        if not ctx.needs_input_grad[1]:  # prompts only
            return None, None, e.vision_backward(d_out)
        if not hasattr(e, "vision_backward_images"):
            raise RuntimeError(f"mudpt_b200: the engine ({type(e).__name__}) has no vision_backward_images: it cannot "
                               "differentiate the vision tower w.r.t. the images")
        dP, d_img = e.vision_backward_images(d_out, want_prompts=ctx.needs_input_grad[2])
        return None, d_img, dP


class TextTowerFn(torch.autograd.Function):
    """f_txt = text_tower(prompts) over the classes registered with Engine.text_set_classes."""

    @staticmethod
    def forward(ctx, engine: Engine, prompts):
        out = engine.text_forward(prompts.detach(), True)
        ctx.engine, ctx.gen = engine, engine.text_gen
        return out

    @staticmethod
    def backward(ctx, d_out):
        e = ctx.engine
        if ctx.gen != e.text_gen:
            raise RuntimeError("mudpt_b200: text backward does not match the latest forward (activations were overwritten)")
        dP, _ = e.text_backward(d_out, False)
        return None, dP


class TextTowerDenseFn(torch.autograd.Function):
    """Module-level API of TextEncoder.forward (trainers/mudpt.py:142-156): arbitrary per-class
    prompt embeddings [C, L, width] in, dense gradient out."""

    @staticmethod
    def setup(engine: Engine, prompts_full, eot, deep_prompts, seq_len, lengths=None) -> torch.Tensor:
        """Registers the per-class prompt embeddings as the class set; returns the prompt stack of the tower call."""
        if lengths is None:  # (engine stand-ins without the ragged form take three arguments)
            engine.text_set_classes(prompts_full.detach(), eot, seq_len)
        else:
            engine.text_set_classes(prompts_full.detach(), eot, seq_len, lengths)
        w = engine.arch["transformer_width"]
        P = torch.zeros(engine.depth, engine.n_ctx, w, device=engine.device, dtype=torch.float32)
        if engine.depth > 1:
            P[1:] = deep_prompts.detach()
        return P

    @staticmethod
    def forward(ctx, engine: Engine, prompts_full, eot, deep_prompts, seq_len, lengths=None):
        P = TextTowerDenseFn.setup(engine, prompts_full, eot, deep_prompts, seq_len, lengths)
        out = engine.text_forward(P, False)
        ctx.engine, ctx.gen = engine, engine.text_gen
        ctx.full_len = prompts_full.shape[1]
        return out

    @staticmethod
    def backward(ctx, d_out):
        e = ctx.engine
        if ctx.gen != e.text_gen:
            raise RuntimeError("mudpt_b200: text backward does not match the latest forward (activations were overwritten)")
        dP, dx0 = e.text_backward(d_out, True)
        d_full = torch.zeros(dx0.shape[0], ctx.full_len, dx0.shape[2], device=dx0.device, dtype=dx0.dtype)
        d_full[:, :dx0.shape[1]] = dx0  # positions past seq_len are dead under the causal mask
        return None, d_full, None, dP[1:], None, None


# Tower calls of the modules: the training forward (activations kept for a backward) only when the result can be
# differentiated, else the forward-only walk -- the same values bitwise, no backward workspace, and a pending backward
# of an earlier training forward stays valid.  (Engine stand-ins without the forward-only entry points take the
# training forward.)
def _differentiable(*inputs) -> bool:
    return torch.is_grad_enabled() and any(x.requires_grad for x in inputs)


def vision_tower(engine: Engine, images, prompts) -> torch.Tensor:
    if _differentiable(images, prompts) or not hasattr(engine, "vision_infer"):
        return VisionTowerFn.apply(engine, images, prompts)
    return engine.vision_infer(images, prompts.detach())


def text_tower(engine: Engine, prompts) -> torch.Tensor:
    if _differentiable(prompts) or not hasattr(engine, "text_infer"):
        return TextTowerFn.apply(engine, prompts)
    return engine.text_infer(prompts.detach(), True)


def text_tower_dense(engine: Engine, prompts_full, eot, deep_prompts, seq_len, lengths=None) -> torch.Tensor:
    if _differentiable(prompts_full, deep_prompts) or not hasattr(engine, "text_infer"):
        return TextTowerDenseFn.apply(engine, prompts_full, eot, deep_prompts, seq_len, lengths)
    return engine.text_infer(TextTowerDenseFn.setup(engine, prompts_full, eot, deep_prompts, seq_len, lengths), False)


class LogitsFn(torch.autograd.Function):
    """logits = exp(logit_scale) * normalize(f_img) @ normalize(f_txt).T (trainers/mudpt.py:178-182)."""

    @staticmethod
    def forward(ctx, engine: Engine, f_img, f_txt):
        logits, _, _, _ = engine.logits_head(f_img.detach(), f_txt.detach(), None, 1.0, False)
        ctx.engine = engine
        ctx.save_for_backward(f_img.detach(), f_txt.detach())
        return logits

    @staticmethod
    def backward(ctx, d_logits):
        f_img, f_txt = ctx.saved_tensors
        d_i, d_t = ctx.engine.logits_backward(f_img, f_txt, d_logits.to(torch.float32))
        return None, d_i, d_t

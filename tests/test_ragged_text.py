"""Ragged text tower: every class prompt runs at its own length (packed rows, variable-length causal attention).

CPU: the lengths and offsets taken from the token ids (with the SOT + n_ctx floor) and the class-cache key.
GPU (`-m gpu`): the variable-length attention kernels against fp32 torch per sequence and bit-identical to the padded
short-sequence kernels on equal lengths; the ragged tower bit-identical to the padded one on equal lengths (every row
kernel with its position arrays) and at rounding level on real ragged lists; the model against the reference fixtures
and the oracle; the CoCoOp dense input gradient; CUDA-graph capture; the C-ABI validation.  Tolerances as stated in
test_gpu_parity.py.
"""
import math

import pytest
import torch

from tests import golden_util as gu

F32_REL = 1e-5
BF16_REL = 5e-3


# ------------------------------------------------------------------------------------------------ CPU
def test_text_lengths_from_token_ids():
    from mudpt_b200.engine import packed_offsets, text_lengths
    tok = torch.zeros(4, 77, dtype=torch.long)
    for c, e in enumerate((6, 2, 11, 4)):  # EOT (the largest id) at position e
        tok[c, :e] = torch.arange(1, e + 1)
        tok[c, e] = 49407
    eot = tok.argmax(-1)
    assert eot.tolist() == [6, 2, 11, 4]
    # n_ctx = 4: every length is at least SOT + 4 prompt rows
    assert text_lengths(eot, "per_class", 77, 5) == (12, [7, 5, 12, 5])
    assert text_lengths(eot, True, 77, 5) == (12, None)
    assert text_lengths(eot, False, 77, 5) == (77, None)
    assert text_lengths(torch.tensor([1, 2]), True, 77, 5) == (5, None)
    assert packed_offsets([7, 5, 12, 5]) == [0, 7, 12, 24, 29]
    with pytest.raises(ValueError, match="per_class"):
        text_lengths(eot, "per-class", 77, 5)


class _RecordingEngine:
    """Stands in for the native engine: records the class set-ups _register_classes asks for."""

    def __init__(self, n_ctx):
        self.device, self.n_ctx, self.class_key, self.calls = torch.device("cpu"), n_ctx, None, []

    def text_set_classes(self, emb, eot, seq_len, lengths=None):
        self.calls.append((tuple(emb.shape), int(seq_len), lengths))


def test_register_classes_cache_key_follows_the_mode():
    c = gu.load("tiny_a")
    model, _ = gu.build_model(c, "cpu")
    eng = _RecordingEngine(c["n_ctx"])
    model._clip_ref[0]._engine = eng
    eot = model.tokenized_prompts.argmax(-1)
    model._register_classes(torch.device("cpu"))
    model._register_classes(torch.device("cpu"))
    assert len(eng.calls) == 1 and eng.calls[0][2] is None
    model.truncate_text_to_eot = "per_class"
    model._register_classes(torch.device("cpu"))
    assert len(eng.calls) == 2
    assert eng.calls[1][2] == [max(int(e) + 1, 1 + c["n_ctx"]) for e in eot.tolist()]
    assert eng.calls[1][1] == max(eng.calls[1][2])
    model._register_classes(torch.device("cpu"))
    assert len(eng.calls) == 2
    model.truncate_text_to_eot = True
    model._register_classes(torch.device("cpu"))
    assert len(eng.calls) == 3 and eng.calls[2][2] is None


# ------------------------------------------------------------------------------------------------ GPU: attention
def _block_rel(a, b, blocks):
    """Worst relative L2 error over the blocks (lists of index tensors into dim 0 of a / b, each [rows, 64]); the
    denominator of a block whose reference is near zero is floored at 0.25 x RMS x sqrt(n) (tests/gpu_bringup._metrics)."""
    a, b = a.double(), b.double()
    rms = float(b.pow(2).mean().sqrt())
    worst = 0.0
    for blk in blocks:
        x, y = a[blk], b[blk]
        den = max(float(y.norm()), 0.25 * rms * math.sqrt(y.numel()))
        worst = max(worst, float((x - y).norm()) / den)
    return worst


def _attn_ref(qkv, do, lengths, H):
    """fp32 causal attention per sequence: o, lse2 (log2 domain of the scaled scores), dq / dk / dv."""
    d = H * 64
    o, lse, dqkv = [], [], []
    r0 = 0
    for n in lengths:
        x = qkv[r0:r0 + n].float().view(n, 3, H, 64).permute(1, 2, 0, 3).clone().requires_grad_(True)
        q, k, v = x[0], x[1], x[2]
        s = (q @ k.transpose(-1, -2)) * 0.125
        s = s.masked_fill(torch.triu(torch.ones(n, n, dtype=torch.bool, device=s.device), 1), float("-inf"))
        y = torch.softmax(s, -1) @ v  # [H, n, 64]
        y.backward(do[r0:r0 + n].float().view(n, H, 64).transpose(0, 1))
        o.append(y.detach().transpose(0, 1).reshape(n, d))
        lse.append((torch.logsumexp(s.detach(), -1) / math.log(2)).reshape(-1))  # [H, n]
        dqkv.append(x.grad.permute(2, 0, 1, 3).reshape(n, 3 * d))
        r0 += n
    return torch.cat(o), torch.cat(lse), torch.cat(dqkv)


def _varlen(lib, qkv, do, off, S, max_len, H, guard=16):
    """Forward and backward through the C ABI into NaN-filled buffers with `guard` spare rows after the packed outputs."""
    from mudpt_b200 import _lib
    M, d = qkv.shape[0], H * 64
    dev = qkv.device
    st = _lib.stream_ptr(dev)
    o = torch.full((M + guard, d), float("nan"), device=dev, dtype=torch.bfloat16)
    lse = torch.full((M * H + guard * H,), float("nan"), device=dev)
    dqkv = torch.full((M + guard, 3 * d), float("nan"), device=dev, dtype=torch.bfloat16)
    _lib.check(lib.mudpt_attention_varlen_forward(qkv.data_ptr(), o.data_ptr(), lse.data_ptr(), off.data_ptr(), S, max_len, H, st))
    _lib.check(lib.mudpt_attention_varlen_backward(qkv.data_ptr(), do.data_ptr(), lse.data_ptr(), dqkv.data_ptr(), off.data_ptr(), S,
                                                   max_len, H, st))
    torch.cuda.synchronize()
    return o, lse, dqkv


@pytest.mark.gpu
@pytest.mark.parametrize("H", [8, 12])
def test_varlen_attention_mixed_lengths(H):
    from mudpt_b200 import _lib
    from mudpt_b200.engine import packed_offsets
    lib = _lib.load()
    torch.manual_seed(H)
    lengths = [17, 1, 77, 3, 64, 16, 32, 15]
    off_l = packed_offsets(lengths)
    M, d, S = off_l[-1], H * 64, len(lengths)
    off = torch.tensor(off_l, dtype=torch.int32, device="cuda")
    qkv = torch.randn(M, 3 * d, device="cuda").bfloat16()
    do = torch.randn(M, d, device="cuda").bfloat16()
    o, lse, dqkv = _varlen(lib, qkv, do, off, S, max(lengths), H)
    # guard bands: nothing written past the packed rows / the M * H statistics
    assert torch.isnan(o[M:].float()).all() and torch.isnan(lse[M * H:]).all() and torch.isnan(dqkv[M:].float()).all()
    o, lse, dqkv = o[:M], lse[:M * H], dqkv[:M]
    assert not torch.isnan(o.float()).any() and not torch.isnan(lse).any() and not torch.isnan(dqkv.float()).any()
    o_ref, lse_ref, dqkv_ref = (t.cpu() for t in _attn_ref(qkv, do, lengths, H))
    o, lse, dqkv = o.float().cpu(), lse.cpu(), dqkv.float().cpu()
    rows = [torch.arange(off_l[s], off_l[s + 1]) for s in range(S)]
    blocks_o = [(r.view(-1, 1), torch.arange(h * 64, h * 64 + 64).view(1, -1)) for r in rows for h in range(H)]
    assert _block_rel(o, o_ref, blocks_o) <= BF16_REL
    assert float((lse - lse_ref).abs().max()) <= 1e-4
    for part in range(3):
        blocks = [(r.view(-1, 1), torch.arange(part * d + h * 64, part * d + h * 64 + 64).view(1, -1)) for r in rows for h in range(H)]
        assert _block_rel(dqkv, dqkv_ref, blocks) <= BF16_REL, ("qkv"[part], H)


@pytest.mark.gpu
@pytest.mark.parametrize("L", [9, 37, 77, 128])
def test_varlen_attention_equal_lengths_bit_identical_to_short_kernels(L):
    from mudpt_b200 import _lib
    lib = _lib.load()
    torch.manual_seed(L)
    S, H = 6, 8
    M, d = S * L, H * 64
    st = _lib.stream_ptr(torch.device("cuda"))
    qkv = torch.randn(M, 3 * d, device="cuda").bfloat16()
    do = torch.randn(M, d, device="cuda").bfloat16()
    o1 = torch.zeros(M, d, device="cuda", dtype=torch.bfloat16)
    lse1 = torch.zeros(S, H, L, device="cuda")
    dsum = torch.zeros(S, H, L, device="cuda")
    dqkv1 = torch.zeros(M, 3 * d, device="cuda", dtype=torch.bfloat16)
    lib.mudpt_set_attention_tc(0)  # the short kernels at every length (by default 65..80 tokens take the tcgen05 backward)
    try:
        _lib.check(lib.mudpt_attention_forward(qkv.data_ptr(), o1.data_ptr(), lse1.data_ptr(), S, L, H, 1, st))
        _lib.check(lib.mudpt_attention_backward(qkv.data_ptr(), o1.data_ptr(), do.data_ptr(), lse1.data_ptr(), dsum.data_ptr(),
                                                dqkv1.data_ptr(), S, L, H, 1, st))
        torch.cuda.synchronize()
    finally:
        lib.mudpt_set_attention_tc(1)
    off = torch.arange(0, M + 1, L, dtype=torch.int32, device="cuda")
    o2, lse2, dqkv2 = _varlen(lib, qkv, do, off, S, L, H)
    assert torch.equal(o1, o2[:M]) and torch.equal(lse1.flatten(), lse2[:M * H]) and torch.equal(dqkv1, dqkv2[:M])


# ------------------------------------------------------------------------------------------------ GPU: tower and model
def _text_inputs(model):
    """Tower inputs of the model's whole class list: embeddings, EOT positions, the prompt stack, per-class lengths."""
    from mudpt_b200.engine import text_lengths
    pl = model.mudpt_prompt_learner
    emb = torch.cat([pl.token_prefix, torch.zeros(pl.n_cls, pl.n_ctx, pl.ctx_dim, device=pl.token_prefix.device),
                     pl.token_suffix], dim=1).float()
    eot = model.tokenized_prompts.argmax(-1)
    with torch.no_grad():
        _, P_t = model.prompt_stacks()
    _, lengths = text_lengths(eot, "per_class", emb.shape[1], 1 + pl.n_ctx)
    return emb, eot, P_t.contiguous(), lengths


def _tower(eng, emb, eot, P_t, d_f, seq_len, lengths=None, dx0=False):
    eng.text_set_classes(emb, eot, seq_len, lengths)
    f = eng.text_forward(P_t).clone()
    dP, d0 = eng.text_backward(d_f, dx0)
    torch.cuda.synchronize()
    return f, dP.clone(), d0


def _set_options(eng, prune, gb):
    from mudpt_b200 import _lib
    _lib.check(eng.lib.mudpt_set_option(eng.h, b"prune", prune), eng.h)
    _lib.check(eng.lib.mudpt_set_option(eng.h, b"grad_stream_bf16", gb), eng.h)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["tiny_b", "tiny_d"])
def test_ragged_tower_equal_lengths_bit_identical_to_padded(name):
    """With every class at the same length the packed layout is the padded one: the position / offset forms of the
    splice LayerNorm, the LayerNorm backward window, the splice backward, the positional add and the attention kernels
    must give the padded tower's features, prompt gradients and dense input gradient bit for bit."""
    c = gu.load(name)
    model, _ = gu.build_model(c, "cuda")
    eng = model._engine(torch.device("cuda"))
    emb, eot, P_t, _ = _text_inputs(model)
    L = int(eot.max()) + 3
    torch.manual_seed(0)
    d_f = torch.randn(emb.shape[0], eng.arch["embed_dim"], device="cuda")
    for prune in (1, 0):
        for gb in (1, 0):
            _set_options(eng, prune, gb)
            for dx0 in (False, True):
                a = _tower(eng, emb, eot, P_t, d_f, L, None, dx0)
                b = _tower(eng, emb, eot, P_t, d_f, L, [L] * emb.shape[0], dx0)
                assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]), (prune, gb, dx0)
                if dx0:
                    assert torch.equal(a[2], b[2]), (prune, gb)
    _set_options(eng, 1, 1)
    model.invalidate_cache()


def _build_vitb16(n_cls, kind, seed=0):
    from mudpt_b200 import clip, synthetic as syn
    from mudpt_b200.trainers.mudpt import CustomCLIP
    arch = syn.ARCHS["ViT-B/16"]
    cfg = gu.make_cfg(2, 9, "a photo of a", 224)
    torch.manual_seed(seed)
    clip_model = clip.CLIP(*arch.astuple(), cfg).float()
    clip_model.load_state_dict(syn.synthetic_clip_state_dict(arch, seed), strict=False)
    model = CustomCLIP(cfg, syn.synthetic_classnames(n_cls, kind), clip_model)
    for n, p in model.named_parameters():
        if "prompt_learner" not in n:
            p.requires_grad_("visual_ctx" in n)
    return model.cuda()


def _close(a, b, cos, rel):
    a, b = a.flatten().double(), b.flatten().double()
    c = float((a @ b) / (a.norm() * b.norm()))
    r = float((a - b).norm() / b.norm())
    return c >= cos and r <= rel, (c, r)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["short", "long"])
def test_ragged_tower_matches_padded(kind):
    """"per_class" against the padded tower on the same ViT-B/16-width text tower (12 layers, 300 classes): features
    and prompt gradients agree at rounding level under every combination of prune and grad_stream_bf16 (the two
    run GEMMs of different row counts, so bf16 roundings downstream differ)."""
    model = _build_vitb16(300, kind)
    eng = model._engine(torch.device("cuda"))
    emb, eot, P_t, lengths = _text_inputs(model)
    if kind == "long":
        assert max(lengths) > min(lengths) + 4
    torch.manual_seed(1)
    d_f = torch.randn(emb.shape[0], eng.arch["embed_dim"], device="cuda") * 1e-2
    for prune in (1, 0):
        for gb in (1, 0):
            _set_options(eng, prune, gb)
            fp, dpp, _ = _tower(eng, emb, eot, P_t, d_f, max(lengths))
            fr, dpr, _ = _tower(eng, emb, eot, P_t, d_f, 0, lengths)
            ok, m = _close(fr, fp, 0.99999, 5e-3)
            assert ok, ("features", prune, gb, m)
            ok, m = _close(dpr, dpp, 0.9999, 2e-2)
            assert ok, ("prompt gradient", prune, gb, m)
    _set_options(eng, 1, 1)
    model.invalidate_cache()


def _check_vs_golden(model, c):
    from tests.gpu_bringup import _metrics
    from oracle import mudpt_oracle as orc
    g = c["golden"]
    image, labels = c["image"].cuda(), c["labels"].cuda()
    model.zero_grad(set_to_none=True)
    loss, logits = model.forward_backward(image, labels)
    torch.cuda.synchronize()
    assert abs(float(loss) - float(g["loss"])) <= 0.02
    m = _metrics(logits.detach().cpu(), torch.from_numpy(g["logits"]))
    assert m["max_abs"] <= 0.05, m
    assert orc.top1_agreement(logits.detach().cpu(), torch.from_numpy(g["logits"]), m["max_abs"])["margin_aware"] >= 0.995
    params = dict(model.named_parameters())
    for k in orc.TRAINABLE:
        ref = torch.from_numpy(g["grad/" + k])
        if ref.numel() and float(ref.norm()) > 0:
            mm = orc.metrics(params[k].grad.detach().cpu(), ref)
            assert mm["cos"] >= 0.999 and mm["rel_l2"] <= 0.05, (k, mm)
    with torch.no_grad():
        prompts, shared, text_deep, t2v = model.mudpt_prompt_learner()
        _, v2t = model.image_encoder(image, shared, t2v)
        f_txt = model.text_encoder(prompts, model.tokenized_prompts, text_deep + v2t)
    assert _metrics(f_txt.cpu(), torch.from_numpy(g["text_features"]))["cos"] >= 0.999


@pytest.mark.gpu
@pytest.mark.parametrize("name", gu.TINY + ["vitb16_cfg1"])
def test_per_class_model_vs_reference_golden(name):
    c = gu.load(name)
    model, _ = gu.build_model(c, "cuda")
    model.truncate_text_to_eot = "per_class"
    model.text_encoder.truncate_to_eot = "per_class"
    _check_vs_golden(model, c)


@pytest.mark.gpu
@pytest.mark.parametrize("name", gu.COCOOP)
def test_per_class_cocoop_vs_reference_golden(name):
    from oracle import mudpt_oracle as orc
    c = gu.load_cocoop(name)
    g = c["golden"]
    model, _ = gu.build_cocoop_model(c, "cuda")
    model.text_encoder.truncate_to_eot = "per_class"
    image, labels = c["image"].cuda(), c["labels"].cuda()
    model.train()
    model.zero_grad(set_to_none=True)
    loss = model(image, labels)
    loss.backward()
    model.eval()
    with torch.no_grad():
        logits = model(image)
    torch.cuda.synchronize()
    assert abs(float(loss) - float(g["loss"])) <= 0.02
    assert float((logits.cpu() - torch.from_numpy(g["logits"])).abs().max()) <= 0.05
    for n, p in model.named_parameters():
        if p.requires_grad:
            m = orc.metrics(p.grad.cpu(), torch.from_numpy(g["grad/" + n]))
            assert m["cos"] >= 0.999 and m["rel_l2"] <= 0.05, (n, m)


@pytest.mark.gpu
def test_per_class_headline_per_rank_shape_long_names_vs_oracle():
    """B = 32 images x C = 125 classes with long names, "per_class", against the CPU oracle."""
    from mudpt_b200 import synthetic as syn
    from oracle import mudpt_oracle as orc
    from tests.test_gpu_parity import _model_and_oracle_sd
    model, sd, arch = _model_and_oracle_sd("ViT-B/16", syn.synthetic_classnames(125, "long"), 2, 9, "a photo of a")
    image = syn.synthetic_images(32, arch.image_resolution, seed=7)
    labels = syn.synthetic_labels(32, 125, seed=7)
    ref = orc.forward_backward(sd, image, model.tokenized_prompts, labels)
    model = model.cuda()
    model.truncate_text_to_eot = "per_class"
    model.zero_grad(set_to_none=True)
    loss, logits = model.forward_backward(image.cuda(), labels.cuda())
    torch.cuda.synchronize()
    assert abs(float(loss) - float(ref["loss"])) <= 0.02
    err = float((logits.cpu() - ref["logits"]).abs().max())
    assert err <= 0.05
    assert orc.top1_agreement(logits.cpu(), ref["logits"], err)["margin_aware"] >= 0.995
    params = dict(model.named_parameters())
    for k in orc.TRAINABLE:
        m = orc.metrics(params[k].grad.cpu(), ref["grads"][k])
        assert m["cos"] >= 0.999 and m["rel_l2"] <= 0.05, (k, m)


@pytest.mark.gpu
def test_cocoop_dense_input_gradient_ragged():
    """CoCoOp's text encoder returns the gradient of its [N, 77, d] prompt embeddings: with "per_class" it is exactly
    zero past each sequence's length and equals the padded tower's inside it (rounding level)."""
    c = gu.load_cocoop("cocoop_tiny_a")
    model, _ = gu.build_cocoop_model(c, "cuda")
    enc = model.text_encoder
    torch.manual_seed(3)
    tok = model.tokenized_prompts.repeat(2, 1)
    prompts = torch.randn(tok.shape[0], tok.shape[1], enc.ln_final.weight.shape[0], device="cuda") * 0.02
    d_f = torch.randn(tok.shape[0], enc.text_projection.shape[1], device="cuda")
    grads = {}
    for mode in (True, "per_class"):
        enc.truncate_to_eot = mode
        p = prompts.clone().requires_grad_(True)
        (enc(p, tok) * d_f).sum().backward()
        grads[mode] = p.grad
    torch.cuda.synchronize()
    n_ctx = model._clip_ref[0].engine().n_ctx
    lengths = [max(int(e) + 1, 1 + n_ctx) for e in tok.argmax(-1).tolist()]
    gp, gr = grads[True], grads["per_class"]
    for s, n in enumerate(lengths):
        assert not gr[s, n:].any(), s
        ok, m = _close(gr[s, :n], gp[s, :n], 0.9999, 2e-2)
        assert ok, (s, m)


@pytest.mark.gpu
def test_ragged_tower_cuda_graph_capture():
    """After the first call (which sizes the workspaces) a ragged forward + backward is capturable and replays to the
    same bits."""
    c = gu.load("tiny_c")
    model, _ = gu.build_model(c, "cuda")
    eng = model._engine(torch.device("cuda"))
    emb, eot, P_t, lengths = _text_inputs(model)
    torch.manual_seed(2)
    d_f = torch.randn(emb.shape[0], eng.arch["embed_dim"], device="cuda")
    f0, dp0, _ = _tower(eng, emb, eot, P_t, d_f, 0, lengths)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        eng.text_forward(P_t)
        eng.text_backward(d_f)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        f = eng.text_forward(P_t)
        dp, _ = eng.text_backward(d_f)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(f, f0) and torch.equal(dp, dp0)
    model.invalidate_cache()


@pytest.mark.gpu
def test_set_classes_ragged_validation():
    c = gu.load("tiny_a")
    model, _ = gu.build_model(c, "cuda")
    eng = model._engine(torch.device("cuda"))
    emb, eot, _, lengths = _text_inputs(model)
    n_ctx = c["n_ctx"]
    bad = list(lengths)
    bad[1] = n_ctx  # shorter than SOT + n_ctx
    with pytest.raises(RuntimeError, match=r"len\[1\]=%d outside" % n_ctx):
        eng.text_set_classes(emb, eot, 0, bad)
    bad = list(lengths)
    bad[0] = emb.shape[1] + 1  # longer than the embeddings
    with pytest.raises(RuntimeError, match=r"len\[0\]=%d outside" % (emb.shape[1] + 1)):
        eng.text_set_classes(emb, eot, 0, bad)
    bad = list(lengths)
    bad[2] = int(eot[2])  # EOT not inside the sequence
    if bad[2] >= 1 + n_ctx:
        with pytest.raises(RuntimeError, match=r"eot\[2\]=%d outside len" % int(eot[2])):
            eng.text_set_classes(emb, eot, 0, bad)
    model.invalidate_cache()

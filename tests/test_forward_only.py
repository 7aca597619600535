"""Forward-only towers (mudpt_vision_infer / mudpt_text_infer) and the QuickGELU-only GEMM epilogues (modes 12 / 13).

Every comparison here is bitwise: the forward-only walk runs the training walk's kernel sequence, and its c_fc epilogue
writes exactly what out1 of modes 3 / 8 writes.  GPU only (`-m gpu`).
"""
import math

import pytest
import torch

from tests import golden_util as gu

GUARD = 8
EPI_GELU, EPI_LN_GELU, EPI_GELU_ONLY, EPI_LN_GELU_ONLY = 3, 8, 12, 13


# ------------------------------------------------------------------------------------------------ fixtures
def _vitb16(n_cls, kind="short", arch_name="ViT-B/16", seed=0):
    """MuDPT CustomCLIP on synthetic weights (n_ctx 2, depth 9), on the GPU."""
    from mudpt_b200 import clip, synthetic as syn
    from mudpt_b200.trainers.mudpt import CustomCLIP
    arch = syn.ARCHS[arch_name]
    cfg = gu.make_cfg(2, 9, "a photo of a", arch.image_resolution, arch_name)
    torch.manual_seed(seed)
    clip_model = clip.CLIP(*arch.astuple(), cfg).float()
    clip_model.load_state_dict(syn.synthetic_clip_state_dict(arch, seed), strict=False)
    model = CustomCLIP(cfg, syn.synthetic_classnames(n_cls, kind), clip_model)
    for n, p in model.named_parameters():
        if "prompt_learner" not in n:
            p.requires_grad_("visual_ctx" in n)
    return model.cuda()


def _cocoop(n_cls, seed=0):
    from mudpt_b200 import clip, synthetic as syn
    from mudpt_b200.trainers.cocoop import CustomCLIP
    arch = syn.ARCHS["ViT-B/16"]
    cfg = gu.make_cocoop_cfg(4, "a photo of a", 224)
    torch.manual_seed(seed)
    clip_model = clip.CLIP(*arch.astuple(), None).float()
    clip_model.load_state_dict(syn.synthetic_clip_state_dict(arch, seed), strict=False)
    model = CustomCLIP(cfg, syn.synthetic_classnames(n_cls), clip_model, tokenizer=syn.synthetic_tokenize)
    for n, p in model.named_parameters():
        if "prompt_learner" not in n:
            p.requires_grad_(False)
    return model.cuda()


def _stacks(model):
    with torch.no_grad():
        P_v, P_t = model.prompt_stacks()
    return P_v.contiguous(), P_t.contiguous()


def _text_inputs(model, C=None, L=None, seed=0):
    """(emb [C, 77, d], eot [C]) of the model's classes, or (C given) C random classes with EOT below L."""
    pl = model.mudpt_prompt_learner
    if C is None:
        emb = torch.cat([pl.token_prefix, torch.zeros(pl.n_cls, pl.n_ctx, pl.ctx_dim, device="cuda"), pl.token_suffix], 1).float()
        return emb, model.tokenized_prompts.argmax(-1)
    g = torch.Generator().manual_seed(seed)
    emb = (torch.randn(C, 77, pl.ctx_dim, generator=g) * 0.02).cuda()
    eot = torch.randint(1 + pl.n_ctx, L, (C,), generator=g)
    return emb, eot


def _opt(eng, name, value):
    from mudpt_b200 import _lib
    _lib.check(eng.lib.mudpt_set_option(eng.h, name.encode(), value), eng.h)


def _images(B, seed=1, size=224):
    from mudpt_b200 import synthetic as syn
    return syn.synthetic_images(B, size, seed=seed).cuda()


# ------------------------------------------------------------------------------------------------ 1. GEMM
@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(6368, 3072, 768), (9625, 2048, 512), (77000, 2048, 512), (32, 2048, 512)])
@pytest.mark.parametrize("stream_k", [0, 1])
def test_gelu_only_epilogues_bitwise_out1(shape, stream_k):
    """Mode 12 = out1 of mode 3 and mode 13 = out1 of mode 8, bit for bit, whole tiles and forced stream-K; every output
    element written (NaN start), 8 guard rows after each output untouched."""
    from mudpt_b200 import _lib
    from tests.gpu_bringup import _gemm_fused
    lib, st = _lib.load(), _lib.stream_ptr(torch.device("cuda"))
    M, N, K = shape
    torch.manual_seed(M + N)
    bf = torch.bfloat16
    x = torch.randn(M, K, device="cuda") * 1.3 + 0.2
    A = x.to(bf)
    W = torch.randn(N, K, device="cuda") * K ** -0.5
    gamma, beta, bias = 1 + 0.2 * torch.randn(K, device="cuda"), 0.2 * torch.randn(K, device="cuda"), 0.5 * torch.randn(N, device="cuda")
    Wl, Wlt = torch.empty(N, K, device="cuda", dtype=bf), torch.empty(K, N, device="cuda", dtype=bf)
    bl, cs, sb = torch.empty(N, device="cuda"), torch.empty(N, device="cuda"), torch.empty(N, 2, device="cuda")
    _lib.check(lib.mudpt_fold_layernorm(W.data_ptr(), gamma.data_ptr(), beta.data_ptr(), bias.data_ptr(), Wl.data_ptr(), Wlt.data_ptr(),
                                        bl.data_ptr(), cs.data_ptr(), sb.data_ptr(), N, K, st))
    xb, stats = torch.empty(M, K, device="cuda", dtype=bf), torch.empty(M, K // 64, 2, device="cuda")
    _lib.check(lib.mudpt_rowstats(x.data_ptr(), xb.data_ptr(), stats.data_ptr(), M, K, st))

    def guarded():
        big = torch.full((M + GUARD, N), float("nan"), device="cuda", dtype=bf)
        return big, big[:M]

    ln = dict(colsum=cs, ln_stats=stats, ln_parts=K // 64, ln_width=K)
    for two, one, a, b, extra in [(EPI_GELU, EPI_GELU_ONLY, A, W.to(bf), dict(bias=bias)),
                                  (EPI_LN_GELU, EPI_LN_GELU_ONLY, xb, Wl, dict(bias=bl, **ln))]:
        bh, h = guarded()
        bg, g = guarded()
        bo, o = guarded()
        _gemm_fused(lib, st, a, b, M, N, K, mode=two, out0=h, out1=g, stream_k=stream_k, **extra)
        _gemm_fused(lib, st, a, b, M, N, K, mode=one, out0=o, stream_k=stream_k, **extra)
        torch.cuda.synchronize()
        assert not torch.isnan(g).any() and not torch.isnan(o).any(), (two, shape)
        assert torch.equal(o.view(torch.int16), g.view(torch.int16)), (one, shape, stream_k)
        assert all(bool(torch.isnan(t[-GUARD:]).all()) for t in (bh, bg, bo)), (one, shape)
    with pytest.raises(RuntimeError, match="needs out0"):
        _gemm_fused(lib, st, A, W.to(bf), M, N, K, mode=EPI_GELU_ONLY, bias=bias)


# ------------------------------------------------------------------------------------------------ 2. towers
@pytest.mark.gpu
@pytest.mark.parametrize("B", [32, 165])
def test_vision_infer_bitwise(B):
    """B = 32 (6,368 rows: stand-alone LayerNorm), B = 165 (32,835 rows: fused), prune 0 and 1."""
    model = _vitb16(10)
    eng = model._engine(torch.device("cuda"))
    P_v, _ = _stacks(model)
    img = _images(B)
    for prune in (1, 0):
        _opt(eng, "prune", prune)
        f = eng.vision_forward(img, P_v).clone()
        gen = eng.vision_gen
        g = eng.vision_infer(img, P_v)
        torch.cuda.synchronize()
        assert torch.equal(f, g), (B, prune)
        assert eng.vision_gen == gen
    _opt(eng, "prune", 1)


@pytest.mark.gpu
def test_vision_infer_bitwise_vitl14():
    """ViT-L/14: 259 tokens, the long-sequence attention kernels."""
    model = _vitb16(4, arch_name="ViT-L/14")
    eng = model._engine(torch.device("cuda"))
    assert eng.arch["vision_width"] == 1024
    P_v, _ = _stacks(model)
    img = _images(6)
    f = eng.vision_forward(img, P_v).clone()
    assert torch.equal(f, eng.vision_infer(img, P_v))


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["padded_125", "padded_1000", "eot", "ragged_long", "dense"])
def test_text_infer_bitwise(case):
    """Padded C = 125 x 77 (9,625 rows, stand-alone LN) and C = 1000 x 77 (77,000 rows, fused), EOT-truncated, ragged
    "per_class" with long names, the dense splice_layer0 = 0 path; prune 0 and 1."""
    from mudpt_b200.engine import text_lengths
    model = _vitb16(125, "long" if case == "ragged_long" else "short")
    eng = model._engine(torch.device("cuda"))
    _, P_t = _stacks(model)
    lengths = None
    if case in ("padded_125", "padded_1000"):
        emb, eot = _text_inputs(model, 125 if case == "padded_125" else 1000, 77)
        L = 77
    else:
        emb, eot = _text_inputs(model)
        L, lengths = text_lengths(eot, "per_class" if case == "ragged_long" else True, 77, 1 + eng.n_ctx)
    eng.text_set_classes(emb, eot, L, lengths)
    splice0 = case != "dense"
    P = P_t.clone()
    if not splice0:
        P[0] = 0
    for prune in (1, 0):
        _opt(eng, "prune", prune)
        f = eng.text_forward(P, splice0).clone()
        gen = eng.text_gen
        g = eng.text_infer(P, splice0)
        torch.cuda.synchronize()
        assert torch.equal(f, g), (case, prune)
        assert eng.text_gen == gen
    _opt(eng, "prune", 1)
    model.invalidate_cache()


@pytest.mark.gpu
def test_plain_towers_infer_bitwise():
    """A plain (n_ctx = 0) handle: CoCoOp's frozen ViT and its dense text tower."""
    model = _cocoop(50)
    eng = model._clip_ref[0].engine()
    assert eng.n_ctx == 0
    img = _images(8)
    empty = torch.zeros(eng.depth, 0, eng.arch["vision_width"], device="cuda")
    f = eng.vision_forward(img, empty).clone()
    assert torch.equal(f, eng.vision_infer(img, empty))
    emb, eot = torch.randn(50, 77, 512, device="cuda") * 0.02, model.tokenized_prompts.argmax(-1)
    eng.text_set_classes(emb, eot, int(eot.max()) + 1)
    P = torch.zeros(eng.depth, 0, 512, device="cuda")
    f = eng.text_forward(P, False).clone()
    assert torch.equal(f, eng.text_infer(P, False))


# ------------------------------------------------------------------------------------------------ 3. non-interference
@pytest.mark.gpu
@pytest.mark.parametrize("ln_fused", [0, 1])
def test_vision_infer_between_forward_and_backward(ln_fused):
    model = _vitb16(10)
    eng = model._engine(torch.device("cuda"))
    _opt(eng, "ln_fused", ln_fused)
    P1, _ = _stacks(model)
    P2 = P1 + 0.05 * torch.randn_like(P1)
    img, img2 = _images(32), _images(48, seed=2)
    d = torch.randn(32, eng.arch["embed_dim"], device="cuda")
    eng.vision_forward(img, P1)
    ref = eng.vision_backward(d).clone()
    eng.vision_forward(img, P1)
    eng.vision_infer(img2, P2)
    got = eng.vision_backward(d)
    torch.cuda.synchronize()
    assert torch.equal(got, ref), ln_fused
    _opt(eng, "ln_fused", -1)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["padded_standalone", "padded_fused", "ragged", "dense"])
def test_text_infer_between_forward_and_backward(case):
    """forward(P1) -> infer(P2) -> backward equals forward(P1) -> backward: d_prompts, and d_x0 on the dense path."""
    from mudpt_b200.engine import text_lengths
    model = _vitb16(125, "long")
    eng = model._engine(torch.device("cuda"))
    _, P1 = _stacks(model)
    P2 = P1 + 0.05 * torch.randn_like(P1)
    emb, eot = _text_inputs(model)
    L, lengths = text_lengths(eot, "per_class" if case == "ragged" else True, 77, 1 + eng.n_ctx)
    _opt(eng, "ln_fused", 1 if case == "padded_fused" else -1)
    eng.text_set_classes(emb, eot, L, lengths)
    splice0, dx0 = case != "dense", case == "dense"
    d = torch.randn(emb.shape[0], eng.arch["embed_dim"], device="cuda")
    eng.text_forward(P1, splice0)
    ref_p, ref_x = (t.clone() if t is not None else None for t in eng.text_backward(d, dx0))
    eng.text_forward(P1, splice0)
    for s in (True, False):
        eng.text_infer(P2, s)
    got_p, got_x = eng.text_backward(d, dx0)
    torch.cuda.synchronize()
    assert torch.equal(got_p, ref_p), case
    if dx0:
        assert torch.equal(got_x, ref_x)
    _opt(eng, "ln_fused", -1)
    model.invalidate_cache()


# ------------------------------------------------------------------------------------------------ 4. memory
def _infer_bytes(eng, tower, S, rows, fused):
    """The inference workspace of DESIGN.md section 3, in bytes, for S sequences / `rows` token rows."""
    a = eng.arch
    e = a["embed_dim"]
    if tower == "vision":
        d, H = a["vision_width"], a["vision_width"] // 64
        stem = 2 * (a["image_resolution"] // a["vision_patch_size"]) ** 2 * ((3 * a["vision_patch_size"] ** 2 + 7) // 8 * 8)
    else:
        d, H, stem = a["transformer_width"], a["transformer_heads"], 0
    per_row = 26 * d + 4 * H + ((4 * d + 16 * (d // 64)) if fused else 0)
    # pruned rows, feature head (gathered rows + split-K partials of the projection), stem patches
    per_seq = 26 * d + 8 * (d // 64) + 4 * (d + max(math.ceil(d / 64) * e, math.ceil(e / 64) * d)) + stem
    sk = 160 * 128 * 256 * 4 + 160 * 16 * 4  # stream-K partial slots + flags
    return rows * per_row + S * per_seq + sk


@pytest.mark.gpu
def test_infer_only_allocates_no_training_workspace():
    """Registering classes and running infer only: no training workspace; the inference workspace is the formula."""
    model = _vitb16(125)
    eng = model._engine(torch.device("cuda"))
    P_v, P_t = _stacks(model)
    emb, eot = _text_inputs(model)
    eng.text_set_classes(emb, eot, 77)
    assert eng.workspace_bytes("text", "train") == 0 and eng.workspace_bytes("text", "infer") == 0
    assert eng.workspace_bytes("text", "input") > 0
    eng.text_infer(P_t)
    eng.vision_infer(_images(32), P_v)
    torch.cuda.synchronize()
    for tower in ("vision", "text"):
        assert eng.workspace_bytes(tower, "train") == 0, tower
    assert eng.workspace_bytes("vision", "input") == 0
    assert eng.workspace_bytes("text", "infer") == _infer_bytes(eng, "text", 125, 125 * 77, False)
    assert eng.workspace_bytes("vision", "infer") == _infer_bytes(eng, "vision", 32, 32 * 199, False)
    model.invalidate_cache()


@pytest.mark.gpu
def test_inference_workspace_at_1000_classes():
    """C = 1000 x 77 (fused LayerNorm): inference bytes <= 1/8 of the training bytes."""
    model = _vitb16(10)
    eng = model._engine(torch.device("cuda"))
    _, P_t = _stacks(model)
    emb, eot = _text_inputs(model, 1000, 77)
    eng.text_set_classes(emb, eot, 77)
    eng.text_infer(P_t)
    eng.text_forward(P_t)
    torch.cuda.synchronize()
    tr, inf = eng.workspace_bytes("text", "train"), eng.workspace_bytes("text", "infer")
    assert inf == _infer_bytes(eng, "text", 1000, 77000, True)
    assert inf * 8 <= tr, (inf, tr, tr / inf)
    print(f"text tower C = 1000 x 77: training workspace {tr / 1e9:.2f} GB, inference {inf / 1e9:.2f} GB ({tr / inf:.1f}x)")
    model.invalidate_cache()


# ------------------------------------------------------------------------------------------------ 5. graph capture
@pytest.mark.gpu
def test_infer_cuda_graph_capture():
    model = _vitb16(125)
    eng = model._engine(torch.device("cuda"))
    P_v, P_t = _stacks(model)
    emb, eot = _text_inputs(model)
    eng.text_set_classes(emb, eot, int(eot.max()) + 1)
    img = _images(16)
    f0, g0 = eng.vision_infer(img, P_v).clone(), eng.text_infer(P_t).clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        eng.vision_infer(img, P_v)
        eng.text_infer(P_t)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        f = eng.vision_infer(img, P_v)
        g = eng.text_infer(P_t)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(f, f0) and torch.equal(g, g0)
    model.invalidate_cache()


# ------------------------------------------------------------------------------------------------ 6. module level
@pytest.mark.gpu
def test_module_eval_paths():
    from mudpt_b200 import synthetic as syn
    c = gu.load("tiny_b")
    model, _ = gu.build_model(c, "cuda")
    eng = model._engine(torch.device("cuda"))
    image = c["image"].cuda()
    labels = c["labels"].cuda()
    # inference() logits = the training entry points' logits
    P_v, P_t = _stacks(model)
    model._register_classes(torch.device("cuda"))
    ref = eng.logits_head(eng.vision_forward(image, P_v), eng.text_forward(P_t), None, 1.0, False)[0].clone()
    model.invalidate_cache()
    gens = (eng.vision_gen, eng.text_gen)
    got = model.inference(image)
    assert torch.equal(got, ref)
    assert (eng.vision_gen, eng.text_gen) == gens
    # model(image) under no_grad = with grad
    with_grad = model(image)
    gens = (eng.vision_gen, eng.text_gen)
    with torch.no_grad():
        no_grad = model(image)
    assert torch.equal(with_grad.detach(), no_grad)
    assert (eng.vision_gen, eng.text_gen) == gens
    # forward -> inference() -> backward: the gradients of forward -> backward
    loss = torch.nn.functional.cross_entropy(model(image), labels)
    loss.backward()
    ref_g = {n: p.grad.clone() for n, p in model.named_parameters() if p.grad is not None}
    assert ref_g
    model.zero_grad(set_to_none=True)
    loss = torch.nn.functional.cross_entropy(model(image), labels)
    model.inference(image[:3])
    loss.backward()
    for n, p in model.named_parameters():
        if n in ref_g:
            assert torch.equal(p.grad, ref_g[n]), n


@pytest.mark.gpu
def test_cocoop_no_grad_forward_equals_grad_forward():
    c = gu.load_cocoop("cocoop_tiny_a")
    model, _ = gu.build_cocoop_model(c, "cuda")
    eng = model._clip_ref[0].engine()
    image = c["image"].cuda()
    model.eval()
    with_grad = model(image)
    gens = (eng.vision_gen, eng.text_gen)
    with torch.no_grad():
        no_grad = model(image)
    torch.cuda.synchronize()
    assert torch.equal(with_grad.detach(), no_grad)
    assert (eng.vision_gen, eng.text_gen) == gens


# ------------------------------------------------------------------------------------------------ 7. CoCoOp evaluation
@pytest.mark.gpu
def test_cocoop_eval_100_images_1000_classes():
    """The MuDPT yaml's test batch (100 images) x 1000 classes = 100,000 text sequences in one forward-only pass.  The
    training-forward footprint at this size is extrapolated from a 2-image run (it would not fit the device)."""
    model = _cocoop(1000)
    eng = model._clip_ref[0].engine()
    model.eval()
    with torch.no_grad():
        model(_images(2))
    torch.cuda.synchronize()
    rows_small = eng.n_classes * eng.text_len
    infer_small = eng.workspace_bytes("text", "infer")
    img = _images(100, seed=3)
    model.train()  # a training forward on 2 images sizes the training workspace for the extrapolation
    model(_images(2), torch.zeros(2, dtype=torch.long, device="cuda")).backward()
    train_per_row = eng.workspace_bytes("text", "train") / rows_small
    model.eval()
    with torch.no_grad():
        logits = model(img)
    torch.cuda.synchronize()
    rows = eng.n_classes * eng.text_len
    assert eng.n_classes == 100 * 1000
    assert logits.shape == (100, 1000) and torch.isfinite(logits).all()
    infer = eng.workspace_bytes("text", "infer")
    train_predicted = train_per_row * rows
    print(f"CoCoOp eval 100 x 1000: {rows} text rows, inference workspace {infer / 1e9:.1f} GB, "
          f"training forward would hold {train_predicted / 1e9:.0f} GB (extrapolated from {infer_small / 1e9:.2f} GB infer at 2 images)")
    assert train_predicted >= 8 * infer
    model.zero_grad(set_to_none=True)

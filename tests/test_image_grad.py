"""Image gradients through the vision tower (mudpt_vision_backward_images, mudpt_col2im, VisionTowerFn into the images,
CustomCLIP.image_gradient).  GPU only (`-m gpu`).

Against the oracle the comparison is per image (cosine >= 0.999, relative L2 <= 5 %, the prompt-gradient bar of the
project); the oracle runs in fp64 on the GPU.  The identities (prompt gradients of the two backward entries, repeat
calls, an evaluation walk in between, graph replay) are bitwise.
"""
import contextlib
import functools

import pytest
import torch
import torch.nn.functional as F

from tests import golden_util as gu

GUARD = 8
COS_MIN, REL_MAX = 0.999, 0.05


# ------------------------------------------------------------------------------------------------ helpers
@contextlib.contextmanager
def _fp64_cuda():
    """The oracle's own torch code in fp64 on the GPU (tensors it creates without a device land there too)."""
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        with torch.device("cuda"):
            yield
    finally:
        torch.set_default_dtype(old)


def _sd64(sd):
    return {k: v.detach().to("cuda", torch.float64) for k, v in sd.items()}


def _per_image(got, ref):
    """worst (cosine, relative L2) over the images of [B, 3, R, R] gradients"""
    g, r = got.double().flatten(1), ref.double().flatten(1)
    cos = (g * r).sum(1) / (g.norm(dim=1) * r.norm(dim=1))
    rel = (g - r).norm(dim=1) / r.norm(dim=1)
    return float(cos.min()), float(rel.max())


def _assert_close(got, ref):
    assert torch.isfinite(got).all()
    cos, rel = _per_image(got, ref)
    assert cos >= COS_MIN and rel <= REL_MAX, (cos, rel)


def _opt(eng, name, value):
    from mudpt_b200 import _lib
    _lib.check(eng.lib.mudpt_set_option(eng.h, name.encode(), value), eng.h)


def _images(B, size, seed=1):
    from mudpt_b200 import synthetic as syn
    return syn.synthetic_images(B, size, seed=seed).cuda()


def _d_feat(B, e, seed=5):
    return torch.randn(B, e, generator=torch.Generator().manual_seed(seed)).cuda()


@functools.lru_cache(maxsize=None)
def _synthetic(arch_name, n_ctx):
    """(engine, oracle state dict with image_encoder.* keys, prompt stack): a plain CLIP (n_ctx 0) or a MuDPT CustomCLIP
    (n_ctx 2, depth 9) on synthetic weights"""
    from mudpt_b200 import clip, synthetic as syn
    arch = syn.ARCHS[arch_name]
    torch.manual_seed(0)
    if n_ctx == 0:
        clip_model = clip.CLIP(*arch.astuple(), None).float()
        clip_model.load_state_dict(syn.synthetic_clip_state_dict(arch, 0), strict=False)
        clip_model = clip_model.cuda()
        eng = clip_model.engine()
        sd = {"image_encoder." + k[len("visual."):]: v for k, v in clip_model.state_dict().items() if k.startswith("visual.")}
        P = torch.zeros(1, 0, arch.vision_width, device="cuda")
        return eng, _sd64(sd), P, clip_model
    from mudpt_b200.trainers.mudpt import CustomCLIP
    cfg = gu.make_cfg(n_ctx, 9, "a photo of a", arch.image_resolution, arch_name)
    clip_model = clip.CLIP(*arch.astuple(), cfg).float()
    clip_model.load_state_dict(syn.synthetic_clip_state_dict(arch, 0), strict=False)
    model = CustomCLIP(cfg, syn.synthetic_classnames(4), clip_model).cuda()
    with torch.no_grad():
        P, _ = model.prompt_stacks()
    eng = model._clip_ref[0].engine()
    return eng, _sd64(model.state_dict()), P.contiguous(), model


def _oracle_d_images(sd64, image, P, d):
    from oracle import mudpt_oracle as orc
    with _fp64_cuda():
        x = image.double().clone().requires_grad_(True)
        f = orc.vision_features_from_stack(sd64, x, P.double())
        return torch.autograd.grad(f, x, d.double())[0]


# ------------------------------------------------------------------------------------------------ 1. col2im
@pytest.mark.gpu
@pytest.mark.parametrize("geom", [(224, 16, 768), (224, 32, 3072), (224, 14, 592)])
def test_col2im_is_fold(geom):
    from mudpt_b200 import _lib
    lib = _lib.load()
    R, p, Kp = geom
    B, npatch, k = 3, (R // p) ** 2, 3 * p * p
    cols = torch.randn(B * npatch, Kp, device="cuda")
    cols[:, k:] = float("nan")  # the padding columns must not be read
    n = B * 3 * R * R
    out = torch.full((n + GUARD,), float("nan"), device="cuda")
    out[n:] = 7.0
    _lib.check(lib.mudpt_col2im(cols.data_ptr(), out.data_ptr(), B, R, p, Kp, _lib.stream_ptr()))
    torch.cuda.synchronize()
    ref = F.fold(cols[:, :k].reshape(B, npatch, k).transpose(1, 2), output_size=R, kernel_size=p, stride=p)
    assert torch.equal(out[:n].view(B, 3, R, R), ref)
    assert torch.equal(out[n:], torch.full((GUARD,), 7.0, device="cuda"))


# ------------------------------------------------------------------------------------------------ 2. against the oracle
@pytest.mark.gpu
@pytest.mark.parametrize("name", gu.TINY)
@pytest.mark.parametrize("prune", [0, 1])
def test_tiny_golden_against_oracle(name, prune):
    c = gu.load(name)
    model, _ = gu.build_model(c)
    eng = model._clip_ref[0].engine()
    _opt(eng, "prune", prune)
    with torch.no_grad():
        P, _ = model.prompt_stacks()
    image = c["image"].cuda()
    d = _d_feat(image.shape[0], c["arch"].embed_dim)
    eng.vision_forward(image, P)
    _, got = eng.vision_backward_images(d, want_prompts=False)
    _assert_close(got, _oracle_d_images(_sd64(c["sd"]), image, P, d))


@pytest.mark.gpu
@pytest.mark.parametrize("case", [("ViT-B/16", 2, 4), ("ViT-B/16", 0, 4), ("ViT-B/32", 2, 2), ("ViT-B/32", 0, 2),
                                  ("ViT-L/14", 2, 2), ("ViT-L/14", 0, 2)])
@pytest.mark.parametrize("prune", [0, 1])
def test_real_widths_against_oracle(case, prune):
    arch_name, n_ctx, B = case
    eng, sd64, P, _ = _synthetic(arch_name, n_ctx)
    _opt(eng, "prune", prune)
    image = _images(B, 224)
    d = _d_feat(B, eng.arch["embed_dim"])
    eng.vision_forward(image, P)
    dP, got = eng.vision_backward_images(d, want_prompts=n_ctx > 0)
    _assert_close(got, _oracle_d_images(sd64, image, P, d))
    _opt(eng, "prune", 1)


@pytest.mark.gpu
def test_fused_layernorm_batch_165():
    """B = 165: 32,835 token rows, the fused-LayerNorm forward.  A per-image gradient depends on its image and its d_f_img
    row only, so three images are checked against the oracle run on those three alone."""
    eng, sd64, P, _ = _synthetic("ViT-B/16", 2)
    B = 165
    image = _images(B, 224, seed=2)
    d = _d_feat(B, eng.arch["embed_dim"], seed=6)
    eng.vision_forward(image, P)
    _, got = eng.vision_backward_images(d, want_prompts=False)
    pick = torch.tensor([0, 82, 164], device="cuda")
    _assert_close(got[pick], _oracle_d_images(sd64, image[pick], P, d[pick]))


# ------------------------------------------------------------------------------------------------ 3. bitwise identities
@pytest.mark.gpu
def test_prompt_gradients_equal_vision_backward():
    eng, _, P, _ = _synthetic("ViT-B/16", 2)
    _opt(eng, "prune", 0)
    _opt(eng, "grad_stream_bf16", 0)
    try:
        image = _images(8, 224)
        d = _d_feat(8, eng.arch["embed_dim"])
        eng.vision_forward(image, P)
        dP_ref = eng.vision_backward(d)
        dP, _ = eng.vision_backward_images(d, want_prompts=True)
        assert torch.equal(dP, dP_ref)
    finally:
        _opt(eng, "prune", 1)
        _opt(eng, "grad_stream_bf16", 1)


@pytest.mark.gpu
@pytest.mark.parametrize("arch_name", ["ViT-B/16", "ViT-B/32"])
def test_repeat_and_evaluation_in_between(arch_name):
    eng, _, P, _ = _synthetic(arch_name, 2)
    image = _images(6, 224)
    d = _d_feat(6, eng.arch["embed_dim"])
    eng.vision_forward(image, P)
    dP0, g0 = eng.vision_backward_images(d)
    dP1, g1 = eng.vision_backward_images(d)
    assert torch.equal(g0, g1) and torch.equal(dP0, dP1)
    eng.vision_forward(image, P)
    eng.vision_infer(_images(11, 224, seed=9), P * 1.5)
    dP2, g2 = eng.vision_backward_images(d)
    assert torch.equal(g0, g2) and torch.equal(dP0, dP2)


# ------------------------------------------------------------------------------------------------ 4. errors and capture
@pytest.mark.gpu
def test_error_paths():
    from mudpt_b200 import _lib
    c = gu.load("tiny_c")
    model, _ = gu.build_model(c)
    eng = model._clip_ref[0].engine()
    with torch.no_grad():
        P, _ = model.prompt_stacks()
    image = c["image"].cuda()
    d = _d_feat(image.shape[0], c["arch"].embed_dim)
    eng.vision_infer(image, P)
    eng.vision_batch = image.shape[0]
    with pytest.raises(RuntimeError, match="no forward pass"):
        eng.vision_backward_images(d)
    eng.vision_forward(image, P)
    _opt(eng, "prune", 0)
    with pytest.raises(RuntimeError, match="no forward pass"):
        eng.vision_backward_images(d)
    _opt(eng, "prune", 1)
    eng.vision_forward(image, P)
    rc = eng.lib.mudpt_vision_backward_images(eng.h, d.data_ptr(), None, None, _lib.stream_ptr())
    assert rc < 0 and b"null argument" in eng.lib.mudpt_last_error(eng.h)
    eng.vision_backward_images(d)  # the handle is still usable


@pytest.mark.gpu
def test_cuda_graph_capture():
    eng, _, P, _ = _synthetic("ViT-B/16", 2)
    B = 4
    image = _images(B, 224)
    d = _d_feat(B, eng.arch["embed_dim"])
    eng.vision_forward(image, P)
    eng.vision_backward_images(d)  # allocates
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        f = eng.vision_forward(image, P)
        dP, dI = eng.vision_backward_images(d)
    image.copy_(_images(B, 224, seed=4))
    g.replay()
    torch.cuda.synchronize()
    f_ref = eng.vision_forward(image, P)
    dP_ref, dI_ref = eng.vision_backward_images(d)
    torch.cuda.synchronize()
    assert torch.equal(f, f_ref) and torch.equal(dP, dP_ref) and torch.equal(dI, dI_ref)


# ------------------------------------------------------------------------------------------------ 5. module level
def _oracle_loss_grad(sd, image, tokenized, labels):
    from oracle import mudpt_oracle as orc
    with _fp64_cuda():
        x = image.double().clone().requires_grad_(True)
        out = orc.forward(_sd64(sd), x, tokenized.cuda(), labels.cuda())
        return torch.autograd.grad(out["loss"], x)[0]


@pytest.mark.gpu
@pytest.mark.parametrize("frozen", [False, True])
def test_custom_clip_forward_image_grad(frozen):
    c = gu.load("tiny_a")
    model, _ = gu.build_model(c)
    if frozen:
        for p in model.parameters():
            p.requires_grad_(False)
    image = c["image"].cuda().requires_grad_(True)
    labels = c["labels"].cuda()
    loss = F.cross_entropy(model(image), labels)
    (g,) = torch.autograd.grad(loss, image)
    _assert_close(g, _oracle_loss_grad(c["sd"], c["image"].cuda(), c["tokenized"], c["labels"]))
    if frozen:
        assert model._clip_ref[0].engine().workspace_bytes("text", "train") == 0


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["tiny_a", "tiny_d"])
def test_image_gradient_fused_step(name):
    c = gu.load(name)
    model, _ = gu.build_model(c)
    image, labels = c["image"].cuda(), c["labels"].cuda()
    loss, logits, g = model.image_gradient(image, labels)
    _assert_close(g, _oracle_loss_grad(c["sd"], image, c["tokenized"], c["labels"]))
    assert torch.equal(logits, model.inference(image))
    assert abs(float(loss) - float(F.cross_entropy(logits, labels))) <= 1e-5 * float(loss)
    assert model._clip_ref[0].engine().workspace_bytes("text", "train") == 0


@pytest.mark.gpu
def test_cocoop_image_grad():
    from oracle import cocoop_oracle as coc
    c = gu.load_cocoop("cocoop_tiny_a")
    model, _ = gu.build_cocoop_model(c)
    model.eval()
    image, labels = c["image"][:2].cuda().requires_grad_(True), c["labels"][:2].cuda()
    loss = F.cross_entropy(model(image), labels)
    (g,) = torch.autograd.grad(loss, image)
    with _fp64_cuda():
        x = c["image"][:2].cuda().double().requires_grad_(True)
        ref = coc.forward(_sd64(c["sd"]), x, c["tokenized"].cuda(), labels)["loss"]
        ref_g = torch.autograd.grad(ref, x)[0]
    _assert_close(g, ref_g)


@pytest.mark.gpu
def test_umudpt_image_grad_is_the_engine_call():
    c = gu.load_variant("umudpt_tiny")
    model, _ = gu.build_variant_model(c)
    eng = model._clip_ref[0].engine()
    image = c["image"].cuda()
    d = _d_feat(image.shape[0], c["arch"].embed_dim)
    x = image.clone().requires_grad_(True)
    vp = model.mudpt_prompt_learner.visual_prompts()
    (g,) = torch.autograd.grad(model.image_encoder(x, vp[:1], vp[1:]), x, d)
    with torch.no_grad():
        P, _ = model.prompt_stacks()
    eng.vision_forward(image, P.contiguous())
    _, ref = eng.vision_backward_images(d, want_prompts=False)
    assert torch.equal(g, ref)

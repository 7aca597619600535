"""The fused l-inf PGD step (mudpt_pgd_linf_update, mudpt_vision_pgd_step), CustomCLIP.pgd_attack and the adversarial
train step CustomCLIP.forward_backward_adversarial.  GPU only (`-m gpu`).

Every comparison is bitwise: the update against the PyTorch formula on the same gradient, the attack against the PyTorch
loop of INTEGRATION.md on image_gradient, and the fused train step against cache_text_features + pgd_attack +
forward_backward(x_adv_norm).
"""
import functools

import pytest
import torch
import torch.nn.functional as F

from tests import golden_util as gu

GUARD = 8
EPS, ALPHA = 4 / 255, 1 / 255
MEAN = (0.48145466, 0.4578275, 0.40821073)
STD = (0.26862954, 0.26130258, 0.27577711)


# ------------------------------------------------------------------------------------------------ helpers
def _chan(v):
    return torch.tensor(v, dtype=torch.float32, device="cuda").view(1, 3, 1, 1)


def _torch_update(g, x_adv, x_clean, eps, alpha, mean=MEAN, std=STD):
    """the PyTorch PGD update, with g = dL/dx_norm (the autograd of the normalisation hands back g / std)"""
    m, s = _chan(mean), _chan(std)
    x = (x_adv + alpha * (g / s).sign()).clamp(x_clean - eps, x_clean + eps).clamp(0, 1)
    return x, (x - m) / s


def _pixels(B, seed=1, R=224):
    return torch.rand(B, 3, R, R, generator=torch.Generator().manual_seed(seed)).cuda()


def _labels(B, C, seed=2):
    return torch.randint(0, C, (B,), generator=torch.Generator().manual_seed(seed)).cuda()


def _d_feat(B, e, seed=5):
    return torch.randn(B, e, generator=torch.Generator().manual_seed(seed)).cuda()


def _cuda_gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


@functools.lru_cache(maxsize=None)
def _model(n_cls, arch_name="ViT-B/16"):
    """MuDPT CustomCLIP (n_ctx 2, depth 9) on synthetic weights with n_cls classes, on the GPU"""
    from mudpt_b200 import clip, synthetic as syn
    from mudpt_b200.trainers.mudpt import CustomCLIP
    arch = syn.ARCHS[arch_name]
    cfg = gu.make_cfg(2, 9, "a photo of a", arch.image_resolution, arch_name)
    torch.manual_seed(0)
    clip_model = clip.CLIP(*arch.astuple(), cfg).float()
    clip_model.load_state_dict(syn.synthetic_clip_state_dict(arch, 0), strict=False)
    model = CustomCLIP(cfg, syn.synthetic_classnames(n_cls), clip_model)
    for n, p in model.named_parameters():
        if "prompt_learner" not in n:
            p.requires_grad_("visual_ctx" in n)
    return model.cuda()


def _plain_clip(arch_name):
    """(engine, empty prompt stack) of a plain CLIP (n_ctx 0) on synthetic weights: a fresh handle"""
    from mudpt_b200 import clip, synthetic as syn
    arch = syn.ARCHS[arch_name]
    torch.manual_seed(0)
    clip_model = clip.CLIP(*arch.astuple(), None).float()
    clip_model.load_state_dict(syn.synthetic_clip_state_dict(arch, 0), strict=False)
    clip_model = clip_model.cuda()
    return clip_model.engine(), torch.zeros(1, 0, arch.vision_width, device="cuda"), clip_model


def _stacks(model):
    with torch.no_grad():
        P_v, _ = model.prompt_stacks()
    return P_v.contiguous()


def _grads(model):
    return {k: p.grad.clone() for k, p in model.named_parameters() if p.requires_grad}


def _zero(model):
    model.zero_grad(set_to_none=True)


def _integration_loop(model, pixels, labels, steps, x0=None):
    """The PGD loop of INTEGRATION.md (image_gradient + PyTorch); returns (x_adv, logits of inference(x_adv_norm))"""
    mean, std = _chan(MEAN), _chan(STD)
    model.eval()
    model.cache_text_features()
    x = pixels.clone() if x0 is None else x0
    for _ in range(steps):
        x.requires_grad_(True)
        xn = (x - mean) / std
        loss, logits, d_xn = model.image_gradient(xn.detach(), labels)
        (d_x,) = torch.autograd.grad(xn, x, d_xn)
        with torch.no_grad():
            x = (x + ALPHA * d_x.sign()).clamp(pixels - EPS, pixels + EPS).clamp(0, 1)
    return x, model.inference((x - mean) / std)


# ------------------------------------------------------------------------------------------------ 1. the update kernel
@pytest.mark.gpu
@pytest.mark.parametrize("geom", [(224, 16, 768), (224, 32, 3072), (224, 14, 592)])
@pytest.mark.parametrize("eps", [EPS, 0.0])
@pytest.mark.parametrize("norm", [(MEAN, STD), ((0.5, 0.25, 0.0), (0.5, 1.5, 3.0))])
def test_update_is_the_torch_formula(geom, eps, norm):
    """mudpt_pgd_linf_update against the formula on F.fold of the same patch gradient: exact-zero and +-subnormal
    gradients, pixels at 0, at 1 and on the eps-box edges; NaN padding columns; guard elements after both outputs."""
    from mudpt_b200 import _lib
    from mudpt_b200.engine import _channels
    lib = _lib.load()
    R, p, Kp = geom
    mean, std = norm
    B, npatch, k = 3, (R // p) ** 2, 3 * p * p
    gen = torch.Generator().manual_seed(R + p)
    g = (torch.randn(B, 3, R, R, generator=gen) * 1e-3).cuda()
    g[0, 0, :6] = 0.0
    g[0, 0, 6:12] = -0.0
    sub = torch.tensor(1e-40).item()
    g[1, 1, :8] = torch.where(torch.rand(8, R, generator=gen) < 0.5, sub, -sub).cuda()
    g[2, 2, :4] = torch.tensor(-1.4e-45).item()  # the smallest subnormal: g / 3 rounds to -0 (no step)
    x_clean = torch.rand(B, 3, R, R, generator=gen).cuda()
    x_clean[0, 1, :8] = 0.0
    x_clean[1, 2, :8] = 1.0
    x_adv = (x_clean + (torch.rand(B, 3, R, R, generator=gen).cuda() * 2 - 1) * eps).clamp(0, 1)
    x_adv[2, 0, :8] = x_clean[2, 0, :8] - eps
    x_adv[2, 1, :8] = x_clean[2, 1, :8] + eps
    x_adv[0, 1, 8:16] = 0.0
    x_adv[1, 2, 8:16] = 1.0
    cols = torch.full((B * npatch, Kp), float("nan"), device="cuda")  # the padding columns must not be read
    cols[:, :k] = F.unfold(g, kernel_size=p, stride=p).transpose(1, 2).reshape(B * npatch, k)
    g_fold = F.fold(cols[:, :k].reshape(B, npatch, k).transpose(1, 2), output_size=R, kernel_size=p, stride=p)
    assert torch.equal(g_fold, g)
    ref_x, ref_n = _torch_update(g_fold, x_adv, x_clean, eps, ALPHA, mean, std)
    n = B * 3 * R * R
    xa = torch.full((n + GUARD,), 7.0, device="cuda")
    xa[:n] = x_adv.flatten()
    xn = torch.full((n + GUARD,), float("nan"), device="cuda")
    xn[n:] = 7.0
    _lib.check(lib.mudpt_pgd_linf_update(cols.data_ptr(), Kp, xa.data_ptr(), x_clean.data_ptr(), xn.data_ptr(), B, R, p,
                                         _channels(mean), _channels(std), eps, ALPHA, _lib.stream_ptr()))
    torch.cuda.synchronize()
    assert torch.equal(xa[:n].view(B, 3, R, R), ref_x)
    assert torch.equal(xn[:n].view(B, 3, R, R), ref_n)
    assert torch.equal(xa[n:], torch.full((GUARD,), 7.0, device="cuda"))
    assert torch.equal(xn[n:], torch.full((GUARD,), 7.0, device="cuda"))
    # the special rows did what the formula says: no step on zero gradients, a full step on subnormal ones
    if eps > 0:
        assert torch.equal(xa[:n].view(B, 3, R, R)[0, 0, :12], x_adv[0, 0, :12])
        assert not torch.equal(xa[:n].view(B, 3, R, R)[1, 1, :8], x_adv[1, 1, :8])


# ------------------------------------------------------------------------------------------------ 2. the tower step
def _pgd_step_case(eng, P, B, seed):
    x_clean = _pixels(B, seed)
    x_adv = (x_clean + (torch.rand(B, 3, 224, 224, generator=torch.Generator().manual_seed(seed + 1)).cuda() * 2 - 1)
             * EPS).clamp(0, 1)
    x_norm = (x_adv - _chan(MEAN)) / _chan(STD)
    d = _d_feat(B, eng.arch["embed_dim"], seed)
    return x_clean, x_adv, x_norm, d


@pytest.mark.gpu
@pytest.mark.parametrize("case", [("ViT-B/16", 2), ("ViT-B/32", 0), ("ViT-L/14", 0)])
def test_vision_pgd_step_is_backward_images_plus_torch(case):
    arch_name, n_ctx = case
    if n_ctx:
        model = _model(4, arch_name)
        eng, P = model._clip_ref[0].engine(), _stacks(model)
    else:
        eng, P, _ = _plain_clip(arch_name)
    B = 6
    x_clean, x_adv, x_norm, d = _pgd_step_case(eng, P, B, 3)
    eng.vision_forward(x_norm, P)
    _, g = eng.vision_backward_images(d, want_prompts=False)
    ref_x, ref_n = _torch_update(g, x_adv, x_clean, EPS, ALPHA)
    eng.vision_pgd_step(d, x_adv, x_clean, x_norm, MEAN, STD, EPS, ALPHA)  # x_norm: the tensor the forward read
    torch.cuda.synchronize()
    assert torch.equal(x_adv, ref_x) and torch.equal(x_norm, ref_n)
    assert not torch.equal(x_adv, x_clean)


@pytest.mark.gpu
@pytest.mark.parametrize("arch_name", ["ViT-B/16", "ViT-B/32"])
def test_pgd_step_memory_is_that_of_image_gradients(arch_name):
    """On a fresh handle: what vision_pgd_step allocates is what vision_backward_images allocates at the same batch
    (ViT-B/32: the patch gradient that does not fit in the QuickGELU transient)."""
    eng, P, _ = _plain_clip(arch_name)
    B = 6
    x_clean, x_adv, x_norm, d = _pgd_step_case(eng, P, B, 4)
    eng.vision_forward(x_norm, P)
    train = eng.workspace_bytes("vision", "train")
    eng.vision_pgd_step(d, x_adv, x_clean, x_norm, MEAN, STD, EPS, ALPHA)
    after_pgd = eng.workspace_bytes("vision", "train")
    eng.vision_forward(x_norm, P)
    eng.vision_backward_images(d, want_prompts=False)
    assert eng.workspace_bytes("vision", "train") == after_pgd
    if arch_name == "ViT-B/32":
        assert after_pgd == train + B * 49 * 3072 * 4
    else:
        assert after_pgd == train


# ------------------------------------------------------------------------------------------------ 3. pgd_attack
@pytest.mark.gpu
@pytest.mark.parametrize("B", [32, 165])
@pytest.mark.parametrize("steps", [1, 5])
@pytest.mark.parametrize("random_start", [False, True])
def test_pgd_attack_is_the_integration_loop(B, steps, random_start):
    model = _model(125)
    pixels, labels = _pixels(B, seed=B), _labels(B, 125)
    x0 = None
    if random_start:
        noise = torch.empty_like(pixels).uniform_(-EPS, EPS, generator=_cuda_gen(9))
        x0 = (pixels + noise).clamp(0, 1)
    ref_x, ref_logits = _integration_loop(model, pixels, labels, steps, x0)
    x_adv, x_norm = model.pgd_attack(pixels, labels, EPS, ALPHA, steps, random_start=random_start, generator=_cuda_gen(9))
    logits = model.inference(x_norm)
    torch.cuda.synchronize()
    assert torch.equal(x_adv, ref_x)
    assert torch.equal(logits, ref_logits)
    assert float((x_adv - pixels).abs().max()) <= EPS * (1 + 1e-6) and not torch.equal(x_adv, pixels)


# ------------------------------------------------------------------------------------------------ 4. the train step
@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(125, True), (1000, False)])  # (classes, EOT-truncated text); 1000: config 2, 77 tokens
@pytest.mark.parametrize("overlap", [True, False])
def test_adversarial_step_is_the_composition(shape, overlap):
    """forward_backward_adversarial = cache_text_features + pgd_attack + forward_backward(x_adv_norm), bitwise: the
    attack between the text training forward and its backward leaves the text tower's saved activations intact."""
    n_cls, truncate = shape
    model = _model(n_cls)
    model.train()
    model.truncate_text_to_eot, model.overlap_towers = truncate, overlap
    B, steps = 32, 3
    pixels, labels = _pixels(B, seed=7), _labels(B, n_cls, seed=8)
    _zero(model)
    model.cache_text_features()
    x_ref, xn_ref = model.pgd_attack(pixels, labels, EPS, ALPHA, steps, random_start=True, generator=_cuda_gen(3))
    loss_r, logits_r = model.forward_backward(xn_ref, labels)
    grads_r = _grads(model)
    loss_r, logits_r = loss_r.clone(), logits_r.clone()
    _zero(model)
    loss, logits, x_adv = model.forward_backward_adversarial(pixels, labels, EPS, ALPHA, steps, random_start=True,
                                                             generator=_cuda_gen(3))
    grads = _grads(model)
    torch.cuda.synchronize()
    model.truncate_text_to_eot, model.overlap_towers = True, True
    assert torch.equal(x_adv, x_ref)
    assert torch.equal(loss, loss_r) and torch.equal(logits, logits_r)
    assert len(grads) == 10
    for k, g in grads.items():
        assert torch.equal(g, grads_r[k]), k


@pytest.mark.gpu
def test_attack_between_steps_changes_nothing():
    model = _model(125)
    model.train()
    a, b = _pixels(32, seed=11), _pixels(32, seed=12)
    labels = _labels(32, 125, seed=13)
    norm = lambda x: (x - _chan(MEAN)) / _chan(STD)  # noqa: E731
    _zero(model)
    model.forward_backward(norm(a), labels)
    _zero(model)
    loss_r, logits_r = model.forward_backward(norm(b), labels)
    loss_r, logits_r, grads_r = loss_r.clone(), logits_r.clone(), _grads(model)
    _zero(model)
    model.forward_backward(norm(a), labels)
    model.pgd_attack(a, labels, EPS, ALPHA, 2)
    _zero(model)
    loss, logits = model.forward_backward(norm(b), labels)
    torch.cuda.synchronize()
    assert torch.equal(loss, loss_r) and torch.equal(logits, logits_r)
    for k, g in _grads(model).items():
        assert torch.equal(g, grads_r[k]), k


# ------------------------------------------------------------------------------------------------ 5. capture and errors
@pytest.mark.gpu
def test_cuda_graph_capture():
    model = _model(4)
    eng, P = model._clip_ref[0].engine(), _stacks(model)
    B = 4
    x_clean, x_adv0, x_norm0, _ = _pgd_step_case(eng, P, B, 21)
    f_txt = torch.randn(16, eng.arch["embed_dim"], generator=torch.Generator().manual_seed(1)).cuda()
    labels = _labels(B, 16)
    x_adv, x_norm = x_adv0.clone(), x_norm0.clone()

    def step():
        f = eng.vision_forward(x_norm, P)
        logits, _, d_i, _ = eng.logits_head(f, f_txt, labels, 1.0 / B, True, text_grad=False)
        eng.vision_pgd_step(d_i, x_adv, x_clean, x_norm, MEAN, STD, EPS, ALPHA)
        return logits

    step()  # allocates
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        logits_g = step()
    out = []
    for run in (graph.replay, step):
        x_adv.copy_(x_adv0)
        x_norm.copy_(x_norm0)
        for _ in range(2):
            r = run()
        torch.cuda.synchronize()
        out.append((x_adv.clone(), x_norm.clone(), (logits_g if r is None else r).clone()))
    for a, b in zip(*out):
        assert torch.equal(a, b)
    assert not torch.equal(out[0][0], x_adv0)


@pytest.mark.gpu
def test_error_paths():
    from mudpt_b200 import _lib
    from mudpt_b200.engine import _channels
    c = gu.load("tiny_c")
    model, _ = gu.build_model(c)
    eng = model._clip_ref[0].engine()
    P = _stacks(model)
    B, R = c["image"].shape[0], c["arch"].image_resolution
    x_clean = _pixels(B, R=R)
    x_adv, x_norm = x_clean.clone(), (x_clean - _chan(MEAN)) / _chan(STD)
    d = _d_feat(B, c["arch"].embed_dim)
    eng.vision_infer(x_norm, P)
    eng.vision_batch = B
    with pytest.raises(RuntimeError, match="no forward pass"):
        eng.vision_pgd_step(d, x_adv, x_clean, x_norm, MEAN, STD, EPS, ALPHA)
    eng.vision_forward(x_norm, P)
    for kw, msg in ((dict(eps=-1e-3), "eps"), (dict(eps=float("inf")), "eps"), (dict(alpha=0.0), "alpha"),
                    (dict(alpha=float("nan")), "alpha"), (dict(std=(0.3, 0.0, 0.3)), "std"),
                    (dict(std=(0.3, -0.2, 0.3)), "std")):
        a = dict(mean=MEAN, std=STD, eps=EPS, alpha=ALPHA)
        a.update(kw)
        with pytest.raises(RuntimeError, match=msg):
            eng.vision_pgd_step(d, x_adv, x_clean, x_norm, **a)
    with pytest.raises(RuntimeError, match="expected shape"):  # a batch other than the forward's
        eng.vision_pgd_step(d, x_adv[:-1].contiguous(), x_clean[:-1].contiguous(), x_norm[:-1].contiguous(), MEAN, STD,
                            EPS, ALPHA)
    rc = eng.lib.mudpt_vision_pgd_step(eng.h, d.data_ptr(), x_adv.data_ptr(), None, x_norm.data_ptr(), _channels(MEAN),
                                       _channels(STD), EPS, ALPHA, _lib.stream_ptr())
    assert rc < 0 and b"null argument" in eng.lib.mudpt_last_error(eng.h)
    torch.cuda.synchronize()
    assert torch.equal(x_adv, x_clean)  # nothing was written by the rejected calls
    eng.vision_pgd_step(d, x_adv, x_clean, x_norm, MEAN, STD, EPS, ALPHA)  # the handle is still usable
    torch.cuda.synchronize()
    assert not torch.equal(x_adv, x_clean)

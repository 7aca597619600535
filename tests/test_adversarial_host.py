"""CPU: the wiring of the fused l-inf PGD attack (CustomCLIP.pgd_attack) and the adversarial train step
(CustomCLIP.forward_backward_adversarial) on an oracle-backed engine stand-in with vision_pgd_step, including UMuDPT and
a gloo world-size-2 step against one process on the concatenated batch."""
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import mudpt_oracle as orc
from tests import golden_util as gu
from tests.oracle_image_engine import OracleImageEngine

EPS, ALPHA, STEPS = 4 / 255, 1 / 255, 3
MEAN = (0.48145466, 0.4578275, 0.40821073)
STD = (0.26862954, 0.26130258, 0.27577711)


class OracleAdversarialEngine(OracleImageEngine):
    """OracleImageEngine with vision_pgd_step: the image gradient of the oracle, then the PyTorch update."""

    def vision_pgd_step(self, d, x_adv, x_clean, x_norm, mean, std, eps, alpha):
        _, g = self.vision_backward_images(d, want_prompts=False)
        m, s = (torch.tensor(v, dtype=torch.float32).view(1, 3, 1, 1) for v in (mean, std))
        x = (x_adv + alpha * (g / s).sign()).clamp(x_clean - eps, x_clean + eps).clamp(0, 1)
        x_adv.copy_(x)
        x_norm.copy_((x - m) / s)


def _attach(model, sd, case):
    eng = OracleAdversarialEngine(sd, case["arch"], case["n_ctx"], case["depth"])
    model._clip_ref[0].engine = lambda device=None: eng
    return eng


def _mudpt(name="tiny_d"):
    c = gu.load(name)
    model, _ = gu.build_model(c, "cpu")
    _attach(model, c["sd"], c)
    return c, model


def _pixels(c, seed=11):
    return torch.rand(c["image"].shape, generator=torch.Generator().manual_seed(seed))


def _torch_loop(model, pixels, labels, steps, x0=None):
    """The PGD loop of INTEGRATION.md on image_gradient"""
    mean, std = (torch.tensor(v).view(1, 3, 1, 1) for v in (MEAN, STD))
    model.cache_text_features()
    x = pixels.clone() if x0 is None else x0.clone()
    for _ in range(steps):
        x.requires_grad_(True)
        xn = (x - mean) / std
        _, _, d_xn = model.image_gradient(xn.detach(), labels)
        (d_x,) = torch.autograd.grad(xn, x, d_xn)
        with torch.no_grad():
            x = (x + ALPHA * d_x.sign()).clamp(pixels - EPS, pixels + EPS).clamp(0, 1)
    return x, (x - mean) / std


def _grads(model):
    return {k: p.grad.clone() for k, p in model.named_parameters() if p.requires_grad}


@pytest.mark.parametrize("random_start", [False, True])
def test_pgd_attack_is_the_torch_loop(random_start):
    c, model = _mudpt()
    pixels, labels = _pixels(c), c["labels"]
    x0 = None
    if random_start:
        noise = torch.empty_like(pixels).uniform_(-EPS, EPS, generator=torch.Generator().manual_seed(5))
        x0 = (pixels + noise).clamp(0, 1)
    x_adv, x_norm = model.pgd_attack(pixels, labels, EPS, ALPHA, STEPS, random_start=random_start,
                                     generator=torch.Generator().manual_seed(5))
    ref, ref_norm = _torch_loop(model, pixels, labels, STEPS, x0)
    assert torch.equal(x_adv, ref) and torch.equal(x_norm, ref_norm)
    assert (x_adv - pixels).abs().max() <= EPS + 1e-7 and not torch.equal(x_adv, pixels)
    assert torch.equal(model.inference(x_norm), model.inference(ref_norm))


@pytest.mark.parametrize("steps", [0, 2])
def test_adversarial_step_is_the_composition(steps):
    c, model = _mudpt()
    pixels, labels = _pixels(c), c["labels"]
    model.cache_text_features()
    x_adv, x_norm = model.pgd_attack(pixels, labels, EPS, ALPHA, steps)
    loss_r, logits_r = model.forward_backward(x_norm, labels)
    grads_r = _grads(model)
    model.zero_grad(set_to_none=True)
    loss, logits, x = model.forward_backward_adversarial(pixels, labels, EPS, ALPHA, steps)
    assert torch.equal(x, x_adv)
    assert torch.allclose(loss, loss_r, rtol=1e-6, atol=0) and torch.allclose(logits, logits_r, rtol=1e-6, atol=1e-6)
    for k, g in _grads(model).items():
        assert torch.allclose(g, grads_r[k], rtol=1e-5, atol=1e-8), k


def test_umudpt_inherits_both_methods():
    c = gu.load_variant("umudpt_tiny")
    model, _ = gu.build_variant_model(c, "cpu")
    _attach(model, {k: v.detach() for k, v in model.state_dict().items()}, c)
    pixels, labels = _pixels(c), c["labels"]
    model.cache_text_features()
    x_adv, x_norm = model.pgd_attack(pixels, labels, EPS, ALPHA, 2)
    ref, _ = _torch_loop(model, pixels, labels, 2)
    assert torch.equal(x_adv, ref)
    loss_r, _ = model.forward_backward(x_norm, labels)
    grads_r = _grads(model)
    model.zero_grad(set_to_none=True)
    loss, _, x = model.forward_backward_adversarial(pixels, labels, EPS, ALPHA, 2)
    assert torch.equal(x, x_adv) and torch.allclose(loss, loss_r, rtol=1e-6, atol=0)
    for k, g in _grads(model).items():
        assert torch.allclose(g, grads_r[k], rtol=1e-5, atol=1e-8), k


def test_engine_without_pgd_step_raises():
    c = gu.load("tiny_d")
    model, _ = gu.build_model(c, "cpu")
    eng = OracleImageEngine(c["sd"], c["arch"], c["n_ctx"], c["depth"])  # image gradients, no vision_pgd_step
    model._clip_ref[0].engine = lambda device=None: eng
    with pytest.raises(RuntimeError, match="vision_pgd_step"):
        model.pgd_attack(_pixels(c), c["labels"], EPS, ALPHA, 1)
    with pytest.raises(RuntimeError, match="vision_pgd_step"):
        model.forward_backward_adversarial(_pixels(c), c["labels"], EPS, ALPHA, 1)


@pytest.mark.parametrize("kw", [dict(eps=-1e-3), dict(eps=math.inf), dict(alpha=0.0), dict(alpha=math.nan),
                                dict(steps=-1), dict(steps=1.5), dict(std=(0.3, 0.0, 0.3)), dict(mean=(0.5, 0.5))])
def test_bad_attack_parameters_raise(kw):
    c, model = _mudpt()
    args = dict(eps=EPS, alpha=ALPHA, steps=1)
    args.update(kw)
    with pytest.raises(ValueError):
        model.pgd_attack(_pixels(c), c["labels"], **args)


# ------------------------------------------------------------------------------------------------ gloo, world size 2
NIMG = 4


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, name, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(2)
    try:
        c = gu.load(name)
        model, _ = gu.build_model(c, "cpu")
        _attach(model, c["sd"], c)
        per = NIMG // world
        pixels, labels = _pixels(c)[rank * per:(rank + 1) * per], c["labels"][rank * per:(rank + 1) * per]
        loss, logits, x_adv = model.forward_backward_adversarial(pixels, labels, EPS, ALPHA, STEPS)
        out[rank] = {"loss": float(loss), "logits": logits.numpy(), "x_adv": x_adv.numpy(),
                     "grads": {k: p.grad.numpy() for k, p in model.named_parameters() if p.requires_grad}}
    finally:
        dist.destroy_process_group()


def test_two_rank_adversarial_step_equals_single_process():
    name = "tiny_d"
    c, model = _mudpt(name)
    pixels, labels = _pixels(c)[:NIMG], c["labels"][:NIMG]
    loss, logits, x_adv = model.forward_backward_adversarial(pixels, labels, EPS, ALPHA, STEPS)
    ref = _grads(model)
    out = mp.Manager().dict()
    mp.spawn(_worker, args=(2, _free_port(), name, out), nprocs=2, join=True)
    assert len(out) == 2
    # the attack is per image; only the loss scale (1 / local batch) differs, so only near-zero gradient components
    # may take another sign
    got = torch.from_numpy(np.concatenate([out[0]["x_adv"], out[1]["x_adv"]], axis=0))
    assert float((got == x_adv).float().mean()) >= 0.999
    assert bool(((got - pixels).abs() <= EPS + 1e-7).all()) and bool(((got >= 0) & (got <= 1)).all())
    np.testing.assert_allclose(np.concatenate([out[0]["logits"], out[1]["logits"]], axis=0), logits.numpy(), atol=2e-4, rtol=0)
    for r in (0, 1):
        np.testing.assert_allclose(out[r]["loss"], float(loss), rtol=1e-5, atol=1e-5)
        for k, g in ref.items():
            if g.numel() and float(g.norm()) > 0:
                m = orc.metrics(torch.from_numpy(out[r]["grads"][k]), g)
                assert m["cos"] > 0.99999 and m["rel_l2"] < 2e-3, (k, r, m)
    for k in out[0]["grads"]:
        np.testing.assert_array_equal(out[0]["grads"][k], out[1]["grads"][k])

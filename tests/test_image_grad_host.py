"""CPU: the autograd wiring of image gradients (VisionTowerFn into the images, the plain ViT, CustomCLIP.image_gradient)
on the oracle-backed engine stand-in (tests/oracle_image_engine.py), against autograd of the oracle itself."""
import pytest
import torch
import torch.nn.functional as F

from oracle import cocoop_oracle as coc
from oracle import mudpt_oracle as orc
from tests import golden_util as gu
from tests.oracle_image_engine import OracleImageEngine, attach


def _close(a, b, tol=1e-4):
    assert a is not None and b is not None
    err = (a - b).norm() / b.norm()
    assert err < tol, float(err)


def _mudpt(name="tiny_a"):
    c = gu.load(name)
    model, _ = gu.build_model(c, "cpu")
    attach(model, c)
    return c, model


def _oracle_image_grad(c, image, labels):
    x = image.clone().requires_grad_(True)
    out = orc.forward(c["sd"], x, c["tokenized"], labels)
    return out["logits"].detach(), out["loss"].detach(), torch.autograd.grad(out["loss"], x)[0]


@pytest.mark.parametrize("frozen", [False, True])
def test_mudpt_forward_differentiates_the_image(frozen):
    c, model = _mudpt()
    if frozen:
        for p in model.parameters():
            p.requires_grad_(False)
    image, labels = c["image"].clone().requires_grad_(True), c["labels"]
    loss = F.cross_entropy(model(image), labels)
    (g,) = torch.autograd.grad(loss, image)
    _close(g, _oracle_image_grad(c, c["image"], labels)[2])


def test_mudpt_image_and_prompt_gradients_together():
    c, model = _mudpt()
    image, labels = c["image"].clone().requires_grad_(True), c["labels"]
    loss = F.cross_entropy(model(image), labels)
    loss.backward()
    _close(image.grad, _oracle_image_grad(c, c["image"], labels)[2])
    ref = orc.forward_backward(c["sd"], c["image"], c["tokenized"], labels)["grads"]
    _close(model.mudpt_prompt_learner.ctx.grad, ref["mudpt_prompt_learner.ctx"], 1e-3)


def test_image_gradient_fused_step():
    c, model = _mudpt()
    labels = c["labels"]
    loss, logits, g = model.image_gradient(c["image"], labels)
    ref_logits, ref_loss, ref_g = _oracle_image_grad(c, c["image"], labels)
    _close(g, ref_g)
    _close(logits, ref_logits, 1e-5)
    assert abs(float(loss) - float(ref_loss)) <= 1e-5 * abs(float(ref_loss))
    assert torch.equal(logits, model.inference(c["image"]))


def test_engine_without_image_backward_raises():
    c, model = _mudpt()
    inner = model._clip_ref[0].engine()

    class WithoutImageBackward:  # an engine stand-in written before image gradients existed
        def __getattr__(self, name):
            if name == "vision_backward_images":
                raise AttributeError(name)
            return getattr(inner, name)

    stand_in = WithoutImageBackward()
    model._clip_ref[0].engine = lambda device=None: stand_in
    image = c["image"].clone().requires_grad_(True)
    loss = F.cross_entropy(model(image), c["labels"])
    with pytest.raises(RuntimeError, match="vision_backward_images"):
        torch.autograd.grad(loss, image)


def test_cocoop_image_gradient_both_paths():
    c = gu.load_cocoop("cocoop_tiny_a")
    model, _ = gu.build_cocoop_model(c, "cpu")
    eng = OracleImageEngine(c["sd"], c["arch"], 0, 1)
    model._clip_ref[0].engine = lambda device=None: eng
    model.eval()
    image = c["image"].clone().requires_grad_(True)
    loss = F.cross_entropy(model(image), c["labels"])
    (g,) = torch.autograd.grad(loss, image)
    x = c["image"].clone().requires_grad_(True)
    ref = coc.forward(c["sd"], x, c["tokenized"], c["labels"])["loss"]
    _close(g, torch.autograd.grad(ref, x)[0])
    # without an image gradient the plain ViT keeps its frozen forward
    with torch.no_grad():
        assert not model.image_encoder(c["image"]).requires_grad


def test_umudpt_image_gradient():
    c = gu.load_variant("umudpt_tiny")
    model, _ = gu.build_variant_model(c, "cpu")
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    eng = OracleImageEngine(sd, c["arch"], c["n_ctx"], c["depth"])
    model._clip_ref[0].engine = lambda device=None: eng
    image = c["image"].clone().requires_grad_(True)
    d = torch.randn(image.shape[0], c["arch"].embed_dim, generator=torch.Generator().manual_seed(3))
    pl = model.mudpt_prompt_learner
    vp = pl.visual_prompts()
    f = model.image_encoder(image, vp[:1], vp[1:])
    (g,) = torch.autograd.grad(f, image, d)
    with torch.no_grad():
        P_v, _ = model.prompt_stacks()
    x = c["image"].clone().requires_grad_(True)
    ref = orc.vision_features_from_stack(sd, x, P_v)
    _close(g, torch.autograd.grad(ref, x, d)[0], 1e-5)

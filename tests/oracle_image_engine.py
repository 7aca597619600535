"""TEST INFRASTRUCTURE: the oracle-backed CPU engine stand-in (tests/fake_engine.py) with image gradients, so that the
autograd wiring into the images (VisionTowerFn, the plain ViT, CustomCLIP.image_gradient) is testable without a GPU.
Never imported by the product."""
import torch

from oracle import mudpt_oracle as orc
from tests.fake_engine import OracleEngine


class OracleImageEngine(OracleEngine):
    """OracleEngine whose vision forward keeps the image as an autograd leaf: vision_backward_images returns its gradient
    (and the prompt gradient), as Engine.vision_backward_images does; logits_head takes text_grad like Engine.logits_head."""

    def vision_forward(self, images, prompts):
        P = prompts.detach().clone().requires_grad_(True)
        X = images.detach().float().clone().requires_grad_(True)
        with torch.enable_grad():
            f = orc.vision_features_from_stack(self.sd, X, P)
        self._v = (P, X, f)
        self.vision_gen += 1
        return f.detach()

    def vision_backward(self, d):
        P, _, f = self._v
        return torch.autograd.grad(f, P, d, retain_graph=True)[0]

    def vision_backward_images(self, d, want_prompts=True):
        P, X, f = self._v
        gP, gX = torch.autograd.grad(f, [P, X], d, retain_graph=True, allow_unused=True)
        if gP is None:  # (no prompt rows)
            gP = torch.zeros_like(P)
        return (gP if want_prompts else None), gX

    def logits_head(self, f_img, f_txt, labels, inv_global_batch, want_grads, text_grad=True):
        logits, loss, di, dt = super().logits_head(f_img, f_txt, labels, inv_global_batch, want_grads)
        return logits, loss, di, (dt if text_grad else None)


def attach(model, case):
    """Route a mudpt_b200 CustomCLIP (built on CPU) through the oracle-backed engine with image gradients."""
    eng = OracleImageEngine(case["sd"], case["arch"], case["n_ctx"], case["depth"])
    model._clip_ref[0].engine = lambda device=None: eng
    return eng

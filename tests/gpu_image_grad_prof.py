"""Image gradients: what the fused attack step costs against the paths around it.

    python tests/gpu_image_grad_prof.py [--out DIR] [--reps N]   (writes DIR/image_grad_prof.json)

MuDPT ViT-B/16 (n_ctx 2, depth 9), 1000 cached classes, frozen prompts, B = 32 and 256:
- image_gradient: CustomCLIP.image_gradient (training vision forward, logits head with labels, backward into the images);
- vision_fwd_prompt_bwd: the same forward and head, then the prompt-only backward (mudpt_vision_backward) -- the
  difference is what the trip to the pixels adds;
- autograd_frozen: torch.autograd.grad(CE(CustomCLIP.forward(image)), image) -- the text tower runs (forward only) on
  every call, which the fused step skips.  (The grad-enabled forward drops the text-feature cache; it is put back after
  each call, so that image_gradient runs on cached features as in an attack loop.)
Medians of the reps, the three alternated in one process; CUDA events around work that ends in a device synchronise.
Then one profiled call of each of the first two: the per-class kernel breakdown (mudpt_profile_end_bound) and its
difference.  The card's name, power limit and clocks are recorded in the same run.
"""
import argparse
import json
import os
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tests.gpu_infer_prof import ab, gpu_info  # noqa: E402
from tests.test_forward_only import _images, _stacks, _vitb16  # noqa: E402

PEAK_TFLOPS, HBM_GBS = 2250.0, 7700.0  # data-sheet dense BF16 and HBM3e figures of one B200 (bounds, not measurements)


def run(res, reps):
    model = _vitb16(1000)
    for p in model.parameters():
        p.requires_grad_(False)
    model.eval()
    P_v, _ = _stacks(model)
    model.cache_text_features()
    f_txt = model._cached_text_features
    eng = model._clip_ref[0].engine()  # the engine of the model's device (cuda:0), the one image_gradient uses
    for B in (32, 256):
        img = _images(B, seed=B)
        assert model._engine(img.device) is eng
        labels = torch.randint(0, 1000, (B,), generator=torch.Generator().manual_seed(B)).cuda()

        def fused():
            model.image_gradient(img, labels)

        def prompt_bwd():
            with torch.no_grad():
                f = eng.vision_forward(img, P_v)
                _, _, d_i, _ = eng.logits_head(f, f_txt, labels, 1.0 / B, True, text_grad=False)
                eng.vision_backward(d_i)

        def autograd_frozen():
            x = img.clone().requires_grad_(True)
            torch.autograd.grad(F.cross_entropy(model(x), labels), x)
            model._cached_text_features = f_txt  # (a grad-enabled forward drops the cache; the next attack step reuses it)

        r = ab({"image_gradient": fused, "vision_fwd_prompt_bwd": prompt_bwd, "autograd_frozen": autograd_frozen}, reps)
        for v in r.values():
            v["images_per_s"] = B / (v["median_ms"] / 1e3)
        r["vision_train_bytes"] = eng.workspace_bytes("vision", "train")
        prof = {}
        for name, fn in (("image_gradient", fused), ("vision_fwd_prompt_bwd", prompt_bwd)):
            torch.cuda.synchronize()
            eng.profile_begin()
            fn()
            prof[name] = eng.profile_end(PEAK_TFLOPS, HBM_GBS)
        r["kernel_classes"] = prof
        r["kernel_classes_added"] = {c: {k: prof["image_gradient"][c][k] - prof["vision_fwd_prompt_bwd"][c][k]
                                         for k in ("ms", "launches", "flops", "bytes")}
                                     for c in prof["image_gradient"]}
        res[f"vitb16_B{B}"] = r
        print(f"B={B}", json.dumps({k: v for k, v in r.items() if k not in ("kernel_classes",)}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.environ.get("TMPDIR", "/tmp"), "mudpt_image_grad_prof"))
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    res = {"gpu": gpu_info()}
    print(res["gpu"], flush=True)
    run(res, a.reps)
    res["gpu_after"] = gpu_info()
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "image_grad_prof.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

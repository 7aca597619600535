"""Adversarial prompt tuning: what the fused l-inf PGD paths cost against the PyTorch compositions they replace.

    python tests/gpu_adversarial_prof.py [--out DIR] [--reps N] [--bench-parent TREE --bench-reps N]
    (writes DIR/adversarial_prof.json)

- evaluation: CustomCLIP.pgd_attack against the PyTorch loop of INTEGRATION.md (image_gradient + ~10 element-wise
  launches per step), 10 steps, B = 32 and 256, MuDPT ViT-B/16 (n_ctx 2, depth 9), 1000 cached classes;
- training: forward_backward_adversarial against the unfused composition cache_text_features + pgd_attack +
  forward_backward(x_adv_norm) at BASELINE config 2 (32 images x 1000 classes), with the text tower at all 77 tokens and
  "per_class", K = 2 and 10 steps; plain forward_backward beside them for scale;
- headline (--bench-parent): `bench.py --gpus 1` of this tree and of TREE (the parent commit's, built), alternated.
Medians of alternated calls; CUDA events around work that ends in a device synchronise.  The card's name, power limit and
clocks are recorded in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tests.gpu_infer_prof import ab, gpu_info  # noqa: E402
from tests.test_forward_only import _vitb16  # noqa: E402

EPS, ALPHA = 4 / 255, 1 / 255
MEAN = (0.48145466, 0.4578275, 0.40821073)
STD = (0.26862954, 0.26130258, 0.27577711)


def _pixels(B, seed):
    return torch.rand(B, 3, 224, 224, generator=torch.Generator().manual_seed(seed)).cuda()


def _labels(B, C, seed):
    return torch.randint(0, C, (B,), generator=torch.Generator().manual_seed(seed)).cuda()


def evaluation(res, model, reps):
    mean, std = (torch.tensor(v, device="cuda").view(1, 3, 1, 1) for v in (MEAN, STD))
    model.eval()
    model.cache_text_features()
    steps = 10
    for B in (32, 256):
        pixels, labels = _pixels(B, B), _labels(B, 1000, B)

        def fused():
            model.pgd_attack(pixels, labels, EPS, ALPHA, steps)

        def torch_loop():
            x = pixels.clone()
            for _ in range(steps):
                x.requires_grad_(True)
                xn = (x - mean) / std
                _, _, d_xn = model.image_gradient(xn.detach(), labels)
                (d_x,) = torch.autograd.grad(xn, x, d_xn)
                with torch.no_grad():
                    x = (x + ALPHA * d_x.sign()).clamp(pixels - EPS, pixels + EPS).clamp(0, 1)

        r = ab({"pgd_attack": fused, "torch_loop": torch_loop}, reps)
        r["speedup"] = r["torch_loop"]["median_ms"] / r["pgd_attack"]["median_ms"]
        res[f"eval_B{B}_K{steps}"] = r
        print(f"eval B={B}", json.dumps(r), flush=True)


def training(res, model, reps):
    model.train()
    B = 32
    pixels, labels = _pixels(B, 7), _labels(B, 1000, 8)
    normed = (pixels - torch.tensor(MEAN, device="cuda").view(1, 3, 1, 1)) / torch.tensor(STD, device="cuda").view(1, 3, 1, 1)
    for mode in (False, "per_class"):
        model.truncate_text_to_eot = mode
        for K in (2, 10):
            def fused():
                model.zero_grad(set_to_none=True)
                model.forward_backward_adversarial(pixels, labels, EPS, ALPHA, K)

            def unfused():
                model.zero_grad(set_to_none=True)
                model.cache_text_features()
                _, xn = model.pgd_attack(pixels, labels, EPS, ALPHA, K)
                model.forward_backward(xn, labels)

            def plain():
                model.zero_grad(set_to_none=True)
                model.forward_backward(normed, labels)

            r = ab({"forward_backward_adversarial": fused, "unfused": unfused, "forward_backward": plain}, reps)
            r["saved_ms"] = r["unfused"]["median_ms"] - r["forward_backward_adversarial"]["median_ms"]
            name = f"train_config2_{'full77' if mode is False else 'per_class'}_K{K}"
            res[name] = r
            print(name, json.dumps(r), flush=True)
    model.truncate_text_to_eot = True


def bench_ab(res, parent, reps, steps, warmup):
    """bench.py --gpus 1 of this tree and of the parent tree, alternated"""
    out = {"this": [], "parent": []}
    for _ in range(reps):
        for name, tree in (("this", ROOT), ("parent", parent)):
            p = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup)],
                               cwd=tree, capture_output=True, text=True)
            line = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
            if p.returncode != 0 or not line:
                raise RuntimeError(f"bench.py in {tree} failed: {p.stderr[-2000:]}")
            out[name].append(json.loads(line[-1]))
    summary = {k: {"value_median": statistics.median(float(r["value"]) for r in v), "values": [float(r["value"]) for r in v],
                   "unit": v[0].get("unit")} for k, v in out.items()}
    summary["ratio_this_over_parent"] = summary["this"]["value_median"] / summary["parent"]["value_median"]
    res["bench_config2_ab"] = summary
    print("bench", json.dumps(summary), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.environ.get("TMPDIR", "/tmp"), "mudpt_adversarial_prof"))
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--bench-parent", default=None, help="a built tree of the parent commit: bench.py A/B against it")
    ap.add_argument("--bench-reps", type=int, default=3)
    ap.add_argument("--bench-steps", type=int, default=30)
    a = ap.parse_args()
    res = {"gpu": gpu_info()}
    print(res["gpu"], flush=True)
    model = _vitb16(1000)
    evaluation(res, model, a.reps)
    training(res, model, a.reps)
    res["gpu_after_timings"] = gpu_info()
    del model
    torch.cuda.empty_cache()
    if a.bench_parent:
        bench_ab(res, a.bench_parent, a.bench_reps, a.bench_steps, 5)
    res["gpu_after"] = gpu_info()
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "adversarial_prof.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

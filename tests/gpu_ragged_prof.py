"""Timing driver: padded against ragged ("per_class") text towers in the fused train step (B200 box).

    python tests/gpu_ragged_prof.py [--steps K] [--warmup W] [--rounds R] [--out FILE]

Workloads: the BASELINE config-2 train step (ViT-B/16, n_ctx 2, depth 9, B = 32 images, C = 1000 classes) with the
short synthetic class names and with synthetic_classnames(1000, "long"), and the config-4 CoCoOp step (B = 2 images x
C = 1000 classes in one text-tower pass).  The two text modes alternate in one process after warm-ups of both, R rounds
of K timed steps each (CUDA events around the step, synchronised); printed: median ms/step per mode, the text-tower rows
each mode runs, and the card's name, power limit and max SM clock.  Test infrastructure only.
"""
from __future__ import annotations

import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _arg(name, dflt):
    return type(dflt)(sys.argv[sys.argv.index(name) + 1]) if name in sys.argv else dflt


def _card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        return "unknown"


def _rows(eot, n_ctx, full_len):
    from mudpt_b200.engine import text_lengths
    padded, _ = text_lengths(eot, True, full_len, 1 + n_ctx)
    _, lengths = text_lengths(eot, "per_class", full_len, 1 + n_ctx)
    return {True: padded * len(lengths), "per_class": sum(lengths)}


def _time(step, set_mode, modes, steps, warmup, rounds):
    import torch
    for m in modes:
        set_mode(m)
        for _ in range(warmup):
            step()
    torch.cuda.synchronize()
    ms = {m: [] for m in modes}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):
        for m in modes:
            set_mode(m)
            step()  # (the class set-up of the mode: not timed)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(steps):
                step()
            e1.record()
            e1.synchronize()
            ms[m].append(e0.elapsed_time(e1) / steps)
    return {m: statistics.median(v) for m, v in ms.items()}


def cfg2(kind, steps, warmup, rounds):
    import torch
    from mudpt_b200 import clip, synthetic as syn
    from mudpt_b200.trainers.mudpt import CustomCLIP
    arch = syn.ARCHS["ViT-B/16"]
    cfg = syn.make_cfg(2, 9, "a photo of a", 224)
    torch.manual_seed(0)
    clip_model = clip.CLIP(*arch.astuple(), cfg).float()
    clip_model.load_state_dict(syn.synthetic_clip_state_dict(arch, 0), strict=False)
    model = CustomCLIP(cfg, syn.synthetic_classnames(1000, kind), clip_model)
    for n, p in model.named_parameters():
        if "prompt_learner" not in n:
            p.requires_grad_("visual_ctx" in n)
    model = model.cuda()
    image = syn.synthetic_images(32, 224, seed=1).cuda()
    label = syn.synthetic_labels(32, 1000, seed=1).cuda()

    def step():
        model.zero_grad(set_to_none=True)
        model.forward_backward(image, label)

    def set_mode(m):
        model.truncate_text_to_eot = m

    ms = _time(step, set_mode, (True, "per_class"), steps, warmup, rounds)
    return ms, _rows(model.tokenized_prompts.argmax(-1), 2, model.tokenized_prompts.shape[1])


def cfg4(steps, warmup, rounds):
    import torch
    from mudpt_b200 import clip, synthetic as syn
    from mudpt_b200.trainers.cocoop import CustomCLIP
    arch = syn.ARCHS["ViT-B/16"]
    cfg = syn.make_cfg(4, 1, "a photo of a", 224)
    cfg.TRAINER["NAME"] = "CoCoOp"
    cfg.TRAINER["COCOOP"] = type(cfg)(N_CTX=4, CTX_INIT="a photo of a", PREC="fp32")
    torch.manual_seed(0)
    clip_model = clip.CLIP(*arch.astuple(), None).float()
    clip_model.load_state_dict(syn.synthetic_clip_state_dict(arch, 0), strict=False)
    model = CustomCLIP(cfg, syn.synthetic_classnames(1000), clip_model, tokenizer=syn.synthetic_tokenize)
    for n, p in model.named_parameters():
        if "prompt_learner" not in n:
            p.requires_grad_(False)
    model = model.cuda().train()
    image = syn.synthetic_images(2, 224, seed=1).cuda()
    label = syn.synthetic_labels(2, 1000, seed=1).cuda()

    def step():
        model.zero_grad(set_to_none=True)
        model(image, label).backward()

    def set_mode(m):
        model.text_encoder.truncate_to_eot = m

    ms = _time(step, set_mode, (True, "per_class"), steps, warmup, rounds)
    rows = _rows(model.tokenized_prompts.argmax(-1).repeat(2), model._clip_ref[0].engine().n_ctx, model.tokenized_prompts.shape[1])
    return ms, rows


def main():
    steps, warmup, rounds = _arg("--steps", 10), _arg("--warmup", 3), _arg("--rounds", 3)
    out = _arg("--out", "")
    lines = [f"card: {_card()}  (name, power limit, max SM clock)",
             f"steps {steps} x rounds {rounds} per mode, warm-up {warmup}; median ms per step; modes alternate in one process"]
    runs = [(f"cfg2 B=32 C=1000 {kind} names", lambda k=kind: cfg2(k, steps, warmup, rounds)) for kind in ("short", "long")]
    runs.append(("cfg4 CoCoOp B=2 x C=1000", lambda: cfg4(steps, warmup, rounds)))
    for tag, fn in runs:
        ms, rows = fn()
        lines.append(f"{tag}: padded {ms[True]:.2f} ms/step ({rows[True]} text rows), per_class {ms['per_class']:.2f} ms/step "
                     f"({rows['per_class']} text rows, {100.0 * (1 - rows['per_class'] / rows[True]):.1f} % fewer), "
                     f"per_class / padded = {ms['per_class'] / ms[True]:.3f}")
        print(lines[-1], flush=True)
    text = "\n".join(lines) + "\n"
    print(text)
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()

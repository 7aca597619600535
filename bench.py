#!/usr/bin/env python
"""bench.py -- MuDPT ViT-B/16 train step throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A "step" = one MuDPT train step of BASELINE config 2: forward + mean cross-entropy + dgrad-only
backward into the 10 prompt tensors + SGD update, batch 32 images per GPU, 1000 classes
(class-sharded over the ranks), ViT-B/16, n_ctx 2, prompt depth 9, synthetic data and random-init
weights (no datasets / checkpoints exist on the box).

One JSON line on stdout (rank 0):
  value   whole-job imgs/s with the step's inputs already resident in HBM, full 77-token text tower
          (the reference formulation, no work skipped)
  e2e     the same metric through the reference-facing call MuDPT.forward_backward(batch) with HOST
          batches: every timed step holds one pinned-host -> device copy of images/labels (issued by
          MuDPT.prefetch(next batch), as a pinned-memory loader does, so it runs under the previous
          step) and the read-back of the step's loss
  eot_truncated   value / e2e with the text tower truncated to max(eot)+1 tokens -- exact under the
          causal mask (SURVEY.md 8c-i), the product default; reported beside, never instead of, the
          full-length numbers
  roofline        the dominant kernel (tcgen05 GEMM): algorithmic FLOPs / CUDA-event time, measured live
          in an instrumented pass of the same step, against the measured sustained bf16 peak
  cpu_baseline    the oracle (fp32 CPU port of the reference path) on a bounded 1/32 sample of the step
`--impl reference` times that CPU path as the main line (the reference itself is pure PyTorch and
cannot travel to the GPU box; oracle/ restates it and is pinned to it by tests/golden).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "train imgs/s MuDPT ViT-B/16 1000-cls"
UNIT = "imgs/s"
BATCH_PER_GPU = 32
N_CLASSES = 1000
N_CTX, DEPTH = 2, 9
ARCH = "ViT-B/16"   # --config 5 switches to ViT-L/14, prompt depth 12 (BASELINE configs[4])


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"bf16_sustained": d.get("bf16_tflops_sustained", 1359.8), "bf16_burst": d.get("bf16_tflops", 1618.5),
                "hbm": d.get("hbm_gbs", 6538.3), "source": "MEASURED_PEAKS.json (of measured)"}
    return {"bf16_sustained": 1400.0, "bf16_burst": 1590.0, "hbm": 6650.0, "source": "B200_PROFILING.md fallback (of fallback)"}


def _gemm_traffic():
    """DRAM bytes per launch of the dominant kernel: dram__bytes_read.sum + dram__bytes_write.sum averaged over EVERY
    tcgen05 GEMM launch of one train step (the population `algorithmic_bytes_per_launch` is averaged over), from the
    committed ncu capture of `bench.py --quick` (profiles/make_step_traffic.py).  The capture names the library build
    it was taken from; a different build gives None (and says so) rather than a stale number."""
    import glob
    import hashlib
    cands = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_step_traffic.json")))
    if not cands:
        return None, "no capture committed"
    d = json.load(open(cands[-1]))
    lib = os.path.join(ROOT, "mudpt_b200", "lib", "libmudpt_b200.so")
    src = hashlib.sha256()
    csrc = os.path.join(ROOT, "mudpt_b200", "csrc")
    for f in ("api.cu", "common.cuh", "gemm.cu", "gemm.h"):  # what decides the step's GEMM launches and their traffic
        src.update(f.encode())
        src.update(open(os.path.join(csrc, f), "rb").read())
    if d.get("csrc_sha256") != src.hexdigest():
        return None, f"{os.path.basename(cands[-1])} was captured from another build of csrc/ (re-run profiles/make_step_traffic.py)"
    return d["avg_traffic_bytes_per_gemm_launch"], os.path.basename(cands[-1])


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0=None, t1=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, power = [], [], set(), []
        for ts, ln in self.lines:
            if t0 is not None and not (t0 - 0.05 <= ts <= t1 + 0.15):
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# CPU path (oracle port of the reference) -- cpu_baseline leg and --impl reference
# ------------------------------------------------------------------------------------------------

def cpu_setup(n_images: int, n_classes: int):
    """Inputs of the oracle (fp32 CPU port of the reference path, pinned to the reference by tests/golden) for a step
    of n_images x n_classes at the headline architecture."""
    from mudpt_b200 import synthetic as syn
    from oracle import mudpt_oracle as orc  # the checker; executed here only as the CPU baseline
    arch = syn.ARCHS["ViT-B/16"]
    names = syn.synthetic_classnames(n_classes)
    tok = syn.synthetic_tokenize(["a photo " + n + "." for n in names])
    ctx_tok = syn.synthetic_tokenize("a photo of a")[0]
    sd = syn.assemble_state_dict(arch, tok, N_CTX, DEPTH, ctx_tok, seed=0)
    image = syn.synthetic_images(n_images, 224, seed=1)
    labels = syn.synthetic_labels(n_images, n_classes, seed=1)
    return orc, sd, image, tok, labels


def cpu_time_steps(steps: int, warmup: int):
    """cpu_baseline leg of the GPU arm: a bounded 1/32 sample of the step (1 image x 32 classes; vision cost is linear
    in images, text cost in classes, so the full 32-image / 1000-class step costs 32 x (1 image + 31.25 classes))."""
    import torch
    orc, sd, image, tok, labels = cpu_setup(1, 32)
    threads = torch.get_num_threads()
    for _ in range(warmup):
        orc.forward_backward(sd, image, tok, labels)
    t0 = time.perf_counter()
    for _ in range(steps):
        orc.forward_backward(sd, image, tok, labels)
    dt = (time.perf_counter() - t0) / max(steps, 1)
    # full step = 32 x sample  ->  imgs/s = 32 / (32 * dt) = 1 / dt
    return {"value": 1.0 / dt, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"1/32 of the step per iteration (1 image x 32 classes, full 77-token text, fp32 torch CPU "
                      f"oracle of the reference path, {threads} threads of {os.cpu_count()} cpus); "
                      f"{steps} timed + {warmup} warm-up iterations, {dt:.2f} s each; imgs/s = 1 / t_iter",
            "s_per_sample_step": dt}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on the box's host cores.  The reference itself
    (pure PyTorch + Dassl, no setup.py) cannot travel to the GPU box; the oracle port restates it (kind: "port").
    With >= 48 GB of free host memory the step is the FULL configuration (32 images x 1000 classes, ~34 GB of fp32
    activations, about a minute per step on 16 cores): 1 warm-up on the 1/32 sample (thread pool, allocator) + at most
    2 timed full steps, so the run ends within a few minutes.  Otherwise the 1/32 sample is timed and scaled."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # other ranks exit 0 without work
    import psutil
    import torch
    torch.set_num_threads(os.cpu_count() or 1)  # torchrun exports OMP_NUM_THREADS=1; use every host thread
    threads = torch.get_num_threads()
    full = psutil.virtual_memory().available >= 48 * 2 ** 30 and os.environ.get("MUDPT_REF_SAMPLE", "0") != "1"
    if full:
        orc, sd, image, tok, labels = cpu_setup(1, 32)
        orc.forward_backward(sd, image, tok, labels)  # warm-up on the sample
        del orc, sd, image, tok, labels
        orc, sd, image, tok, labels = cpu_setup(BATCH_PER_GPU, N_CLASSES)
        steps, warm = max(1, min(args.steps, 2)), 1
        t0 = time.perf_counter()
        for _ in range(steps):
            orc.forward_backward(sd, image, tok, labels)
        dt = (time.perf_counter() - t0) / steps
        value, ms = BATCH_PER_GPU / dt, dt * 1e3
        cb = {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
              "sample": f"the full step ({BATCH_PER_GPU} images x {N_CLASSES} classes, 77-token text, fp32 torch CPU oracle of the "
                        f"reference path, {threads} threads of {os.cpu_count()} cpus): {steps} timed step(s) of {dt:.1f} s after a "
                        f"warm-up on a 1/32 sample", "s_per_step": dt}
    else:
        steps, warm = max(1, min(args.steps, 40)), max(1, min(args.warmup, 3))
        cb = cpu_time_steps(steps, warm)
        value, ms = cb["value"], cb["s_per_sample_step"] * 32 * 1e3
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"MuDPT ViT-B/16 16-shot-shaped train step (BASELINE configs[1]): batch {BATCH_PER_GPU}/GPU, "
                               f"{N_CLASSES} classes, n_ctx {N_CTX}, prompt depth {DEPTH} (CPU fp32 path, one process; does not "
                               "scale with --gpus)", "text_seq_len": 77, "full_configuration": bool(full)},
        "cpu_baseline": cb,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU path
# ------------------------------------------------------------------------------------------------

def build_trainer(device, truncate: bool, n_classes: int = N_CLASSES):
    import torch
    from mudpt_b200 import synthetic as syn
    from mudpt_b200.trainers import mudpt as M
    arch = syn.ARCHS[ARCH]
    cfg = syn.make_cfg(N_CTX, DEPTH, "a photo of a", arch.image_resolution, ARCH)
    torch.manual_seed(0)  # prompt parameters are torch-initialised: identical replicas on every rank
    clip_model = M.clip.CLIP(*arch.astuple(), cfg).float()
    clip_model.load_state_dict(syn.synthetic_clip_state_dict(arch, 0), strict=False)
    trainer = M.MuDPT.__new__(M.MuDPT)
    M.TrainerX.__init__(trainer, None, None, device)
    trainer.cfg = cfg
    trainer.check_cfg(cfg)
    model = M.CustomCLIP(cfg, syn.synthetic_classnames(n_classes), clip_model)
    for n, p in model.named_parameters():  # freeze rule, trainers/mudpt.py:205-212
        if "prompt_learner" not in n:
            p.requires_grad_("visual_ctx" in n)
    model.truncate_text_to_eot = truncate
    model.to(device)
    trainer.model = model
    trainer.optim = M.build_optimizer(model, cfg.OPTIM)
    trainer.sched = M.build_lr_scheduler(trainer.optim, cfg.OPTIM)
    trainer.register_model("MultimodalDeepPromptTuning", model, trainer.optim, trainer.sched)
    trainer.batch_idx, trainer.num_batches = 0, 10 ** 9
    return trainer


def timed_loop(fn, steps, warmup, device, world):
    """W warm-ups, then exactly K steps bracketed by barrier + synchronize, CUDA events on the
    launching stream, max over ranks."""
    import torch
    import torch.distributed as dist
    for i in range(warmup):
        fn(i)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    e0.record()
    for i in range(steps):
        fn(warmup + i)
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(device)
    t1 = time.time()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    return ms, t0, t1


def run_ours(args):
    import torch
    import torch.distributed as dist
    from mudpt_b200 import synthetic as syn
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference)")
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    K, W = args.steps, max(args.warmup, 3)
    B = BATCH_PER_GPU
    NBUF = 8  # 8 distinct batches = 154 MB of inputs > 126 MB L2; the step's activations are GBs

    imgs_host = [syn.synthetic_images(B, 224, seed=100 + rank * NBUF + i).pin_memory() for i in range(NBUF)]
    labs_host = [syn.synthetic_labels(B, N_CLASSES, seed=100 + rank * NBUF + i).pin_memory() for i in range(NBUF)]
    imgs_dev = [t.to(device) for t in imgs_host]
    labs_dev = [t.to(device) for t in labs_host]

    results = {}
    sampler = ClockSampler(local)
    clocks = None
    if args.quick:
        # profiling aid (ncu launch lists): the full-length variant's resident loop only, no JSON contract
        # --classes emulates the per-GPU shapes of an N-rank run on one GPU (1000 / N classes), no NCCL
        trainer = build_trainer(device, False, args.classes)
        labs_dev = [t % args.classes for t in labs_dev]
        if args.no_overlap:
            trainer.model.overlap_towers = False

        def step_q(i):
            trainer.optim.zero_grad()
            trainer.model.forward_backward(imgs_dev[i % NBUF], labs_dev[i % NBUF])
            trainer.optim.step()

        ms, _, _ = timed_loop(step_q, K, W, device, world)
        eng = trainer.model._clip_ref[0].engine(device)
        overlap = trainer.model.overlap_towers
        trainer.model.overlap_towers = False
        eng.profile_begin()
        torch.cuda.synchronize(device)
        for i in range(3):
            step_q(i)
        prof = eng.profile_end()
        trainer.model.overlap_towers = overlap
        if rank == 0:
            print(json.dumps({"quick": True, "ms_per_step": ms / K, "value": B * world / (ms / K * 1e-3), "unit": UNIT,
                              "kernels_ms_per_step": {k: round(v["ms"] / 3, 3) for k, v in prof.items() if v["launches"]},
                              "kernels_us_per_launch": {k: round(v["ms"] * 1e3 / v["launches"], 1) for k, v in prof.items() if v["launches"]},
                              "gemm_tflops": round(prof["gemm"]["flops"] / max(prof["gemm"]["ms"], 1e-9) / 1e9, 1)}))
        if world > 1:
            dist.destroy_process_group()
        return
    batches_host = []
    for variant, truncate in (("full", False), ("eot_truncated", True)):
        trainer = build_trainer(device, truncate)
        model = trainer.model
        eng = model._clip_ref[0].engine(device)
        last = {}

        def step_resident(i):
            trainer.optim.zero_grad()
            out = model.forward_backward(imgs_dev[i % NBUF], labs_dev[i % NBUF])
            if args.dump_outputs:
                last["loss"], last["logits"] = out
            trainer.optim.step()

        def step_e2e(i):
            # the reference-facing call: host batch in, python float out (trainers/mudpt.py:235-261)
            # (prefetch = what a pinned-memory loader does: batch i + 1 is uploaded on a copy stream under step i; every
            # step's timed region still holds one batch upload and the loss read-back)
            if not batches_host:
                batches_host.extend({"img": imgs_host[j], "label": labs_host[j]} for j in range(NBUF))
            trainer.prefetch(batches_host[(i + 1) % NBUF])
            return trainer.forward_backward(batches_host[i % NBUF])

        l0 = eng.launch_count()
        if variant == "full":
            sampler.start()
        ms, t0, t1 = timed_loop(step_resident, K, W, device, world)
        if variant == "full":
            clocks = sampler.stop(t0, t1)
            if args.dump_outputs and rank == 0:  # before any further step overwrites them
                dump_outputs(args.dump_outputs, model, last["loss"], last["logits"])
        launches = (eng.launch_count() - l0) // (K + W)
        ms_e2e, _, _ = timed_loop(step_e2e, K, W, device, world)
        # instrumented pass of the same step: per-kernel-class CUDA-event times
        # (single stream: with the towers overlapped an event pair would also time the other tower's kernels)
        overlap = model.overlap_towers
        model.overlap_towers = False
        eng.profile_begin()
        torch.cuda.synchronize(device)
        for i in range(min(K, 5)):
            step_resident(i)
        pk = _peaks()
        prof = eng.profile_end(pk["bf16_sustained"], pk["hbm"])
        model.overlap_towers = overlap
        nprof = min(K, 5)
        results[variant] = {"model_dict": model.__dict__, "ms": ms / K, "ms_e2e": ms_e2e / K, "launches": launches, "prof": prof, "nprof": nprof,
                            "text_len": eng.text_len, "loss": float(trainer.forward_backward(
                                {"img": imgs_host[0], "label": labs_host[0]})["loss"])}
        del trainer, model, eng
        torch.cuda.empty_cache()

    dist_check = collectives = None
    if world > 1:
        dist_check = sharded_equivalence_check(device, imgs_dev[0], labs_dev[0], world)
        collectives = collective_timings(device, world)
    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    peaks = _peaks()
    full, tr = results["full"], results["eot_truncated"]
    gB = B * world
    g = full["prof"]["gemm"]
    gemm_tflops = g["flops"] / (g["ms"] * 1e-3) / 1e12 if g["ms"] > 0 else 0.0
    # ("gemm" is the sum of the per-GEMM entries "gemm_*": count it once)
    step_prof_ms = sum(v["ms"] for k, v in full["prof"].items() if not k.startswith("gemm_")) / full["nprof"]
    shares = {k: round(v["ms"] / full["nprof"] / step_prof_ms, 4) for k, v in full["prof"].items() if v["ms"] > 0}

    def cat_table(prof, nprof):
        out = {}
        for k, v in prof.items():
            if v["launches"] == 0:
                continue
            us = v["ms"] * 1e3 / v["launches"]
            e = {"launches_per_step": v["launches"] // nprof, "avg_us": round(us, 2), "ms_per_step": round(v["ms"] / nprof, 4)}
            if v["flops"] > 0:
                e["tflops"] = round(v["flops"] / (v["ms"] * 1e-3) / 1e12, 1)
            e["gbs_algorithmic"] = round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1)
            if v.get("bound_ms", 0) > 0:  # time at the bound that applies to each launch (tensor or HBM) / measured time
                e["frac_of_applicable_bound"] = round(v["bound_ms"] / v["ms"], 3)
            out[k] = e
        return out

    h2d = B * 3 * 224 * 224 * 4 + B * 8
    # rank 0 at N=1 only (torchrun pins OMP threads to 1); the oracle sample is the headline architecture's
    cb = cpu_time_steps(3, 1) if (world == 1 and ARCH == "ViT-B/16") else None
    pipe = infer = None
    if world == 1 and ARCH == "ViT-B/16":
        try:
            pipe = input_pipeline_bench(device, peaks)
        except Exception as e:  # an aside to the contract line: never lose the headline over it
            pipe = {"error": f"{type(e).__name__}: {e}"}
        try:
            infer = inference_bench(device)
        except Exception as e:
            infer = {"error": f"{type(e).__name__}: {e}"}
    line = {
        "metric": METRIC if ARCH == "ViT-B/16" else f"train imgs/s MuDPT {ARCH} 1000-cls depth {DEPTH}",
        "value": gB / (full["ms"] * 1e-3), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": full["ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"MuDPT {ARCH} 16-shot-shaped train step (BASELINE configs[{1 if ARCH == 'ViT-B/16' else 4}]): batch {B}/GPU, "
                               f"{N_CLASSES} classes sharded by class over {world} rank(s), n_ctx {N_CTX}, prompt depth {DEPTH}, "
                               "fwd + CE + dgrad-only bwd + SGD step, random-init weights",
                   "global_batch": gB, "classes_per_gpu": -(-N_CLASSES // world), "text_seq_len": full["text_len"],
                   "parallelism": f"dp{world} images x class-sharded text",
                   "l2": f"{NBUF} rotating input batches (154 MB > 126 MB L2); per-step activation working set is several GB",
                   "operands": "bf16 GEMM/attention operands, fp32 accumulate, fp32 residual stream / LN / softmax / loss; the residual "
                               "stream's GRADIENT travels between the LayerNorm backward kernels as bf16 (option grad_stream_bf16)"},
        "e2e": {"value": gB / (full["ms_e2e"] * 1e-3), "unit": UNIT, "ms_per_step": full["ms_e2e"],
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "api": "mudpt_b200.trainers.mudpt.MuDPT.prefetch(next batch) + forward_backward(batch): pinned host batches, each uploaded under the previous step; loss read back every step"},
        "gpu_launches": full["launches"] * K,
        "gpu_launches_per_step": full["launches"],
        "eot_truncated": {"value": gB / (tr["ms"] * 1e-3), "ms_per_step": tr["ms"], "text_seq_len": tr["text_len"],
                          "e2e": {"value": gB / (tr["ms_e2e"] * 1e-3), "ms_per_step": tr["ms_e2e"]},
                          "gpu_launches_per_step": tr["launches"], "kernels": cat_table(tr["prof"], tr["nprof"]),
                          "note": "text tower run on max(eot)+1 tokens: exact under the causal mask (tests), product default"},
        "roofline": {"bound": "tensor", "kernel": "gemm_tn_tcgen05_kernel (all GEMM launches of the step)",
                     "achieved": round(gemm_tflops, 1), "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
                     "frac": round(gemm_tflops / peaks["bf16_sustained"], 4),
                     # the same launches, each against the bound that applies to IT: max(FLOPs / sustained bf16 peak,
                     # algorithmic bytes / measured HBM rate) summed over the launches / their measured time (the K = 512
                     # GEMMs with fp32 or twin bf16 outputs are HBM-bound by their own algorithmic bytes)
                     "frac_of_applicable_bound": round(g.get("bound_ms", 0.0) / g["ms"], 4) if g["ms"] > 0 else None,
                     "traffic": _gemm_traffic()[0],
                     "traffic_source": _gemm_traffic()[1],
                     "algorithmic_bytes_per_launch": g["bytes"] / max(g["launches"], 1),
                     "peak_source": peaks["source"] + ", sustained figure (kernel timed inside a long step)",
                     "launches_per_step": g["launches"] // full["nprof"],
                     "avg_launch_us": round(g["ms"] * 1e3 / max(g["launches"], 1), 2),
                     "flops_per_launch": g["flops"] / max(g["launches"], 1),
                     "share_of_step": shares},
        "kernels": cat_table(full["prof"], full["nprof"]),
        # reference formulation = every row of every block, forward + dgrad (SURVEY.md 8d); executed = what the
        # launches of the step actually compute after the exact work skipping of the last block (CLS / EOT rows only)
        "step_flops_reference_formulation_T": round(reference_step_flops(B, -(-N_CLASSES // world), full["text_len"]) / 1e12, 3),
        "step_flops_executed_T": round((g["flops"] + full["prof"]["attn_fwd"]["flops"] +
                                        full["prof"]["attn_bwd"]["flops"]) / full["nprof"] / 1e12, 3),
        "loss": full["loss"], "loss_eot_truncated": tr["loss"],
        "clocks": clocks,
        "cpu_baseline": cb,
        "input_pipeline": pipe,
        "inference_cfg3": infer,
        "sharded_vs_unsharded": dist_check,
        "collectives_us": collectives,
        # how the head's text-feature exchange ran in the timed step (mudpt_b200/dist.py:PeerExchange)
        "head_exchange": (None if world == 1 else
                          "peer memory over NVLink (own pull kernels after a symmetric-memory barrier)"
                          if full["model_dict"].get("peer_exchange") is not None else "NCCL all_gather / reduce_scatter"),
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()



def dump_outputs(out_dir, model, loss, logits):
    """--dump-outputs: what the last timed step of the headline hands its caller, one float32 .npy per array: the loss,
    rank 0's logits, and for each of the 10 trainable prompt tensors its gradient (grad.<name>) and its value after the
    SGD update (param.<name>).  About 10 MB at ViT-B/16 and 19 MB at ViT-L/14.  The inputs are seeded, so two builds
    run with the same arguments can be compared array by array."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss, "logits": logits}
    for n, p in model.named_parameters():
        if p.requires_grad:
            arrays["grad." + n], arrays["param." + n] = p.grad, p
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def reference_step_flops(batch, classes, text_len):
    """Per-rank FLOPs of one train step in the reference formulation: 12 d^2 MACs per token and block forward, the same
    again for the dgrad (no wgrad: frozen weights), attention 4 L^2 64 per head forward and 2.5 x that backward."""
    from mudpt_b200 import synthetic as syn
    a = syn.ARCHS[ARCH]
    fl = 0.0
    for (S, L, d, layers) in ((batch, (a.image_resolution // a.vision_patch_size) ** 2 + 1 + N_CTX, a.vision_width, a.vision_layers),
                              (classes, text_len, a.transformer_width, a.transformer_layers)):
        M, H = S * L, d // 64
        fl += layers * (2 * 24.0 * M * d * d + 3.5 * 4.0 * S * H * L * L * 64)
    return fl


def sharded_equivalence_check(device, image, label, world):
    """N > 1: the class-sharded step (text tower over C / N classes per rank, all-gather of the text features,
    reduce-scatter of their gradient, all-reduce of the prompt gradients) against the UNSHARDED step on the same
    images (every rank runs all classes; gradients summed over ranks by hand): logits max-abs / cosine, loss and
    the worst gradient cosine.  Not bitwise: the stream-K cut of a GEMM depends on its row count."""
    import torch
    import torch.distributed as dist
    trainer = build_trainer(device, True)
    model = trainer.model
    out = {}
    res = {}
    for mode in ("sharded", "unsharded"):
        model.shard_classes = mode == "sharded"
        model._clip_ref[0].engine(device).class_key = None
        model.zero_grad(set_to_none=True)
        loss, logits = model.forward_backward(image, label)
        grads = [p.grad.detach().clone() for p in model.parameters() if p.requires_grad]
        if mode == "unsharded":  # local-batch mean -> global-batch mean, summed over the ranks
            loss = loss.detach().clone() / world
            dist.all_reduce(loss)
            for g in grads:
                g.div_(world)
                dist.all_reduce(g)
        res[mode] = (float(loss), logits.detach().clone(), grads)
    a, b = res["sharded"], res["unsharded"]
    la, lb = a[1].flatten().double(), b[1].flatten().double()
    out["logits_max_abs"] = float((a[1] - b[1]).abs().max())
    out["logits_cos"] = float((la @ lb) / (la.norm() * lb.norm()))
    out["loss"] = [a[0], b[0]]
    cos = []
    for ga, gb in zip(a[2], b[2]):
        x, y = ga.flatten().double(), gb.flatten().double()
        cos.append(float((x @ y) / (x.norm() * y.norm() + 1e-300)))
    out["grad_cos_min"] = min(cos)
    t = torch.tensor([out["logits_max_abs"], -out["logits_cos"], -out["grad_cos_min"]], device=device, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)  # worst over the ranks
    out["logits_max_abs"], out["logits_cos"], out["grad_cos_min"] = float(t[0]), -float(t[1]), -float(t[2])
    out["ranks"] = world
    del trainer, model
    torch.cuda.empty_cache()
    return out


def collective_timings(device, world, reps=20):
    """Device time (CUDA events, max over ranks) of each collective of the step at its real size: all-gather of the
    text features [C / N, 512] -> [C, 512], reduce-scatter of their gradient, all-reduce of the 1.2 M prompt-gradient
    floats in one bucket, all-reduce of the loss scalar."""
    import torch
    import torch.distributed as dist
    from mudpt_b200 import dist as mdist
    C, e = N_CLASSES, 512
    lo, hi = mdist.shard_bounds(C, dist.get_rank(), world)
    f_loc = torch.randn(hi - lo, e, device=device)
    d_full = torch.randn(C, e, device=device)
    grads = [torch.nn.Parameter(torch.randn(n, device=device)) for n in (1024, 8 * 1024, 393216, 768, 393216, 768, 1536, 12288, 393216, 512)]
    for p in grads:
        p.grad = torch.randn_like(p)
    loss = torch.zeros((), device=device)
    bucket = mdist.FlatGrads(grads)   # what the fused step does: the gradients live in one flat bucket
    ops = {"all_gather_text_features": lambda: mdist.all_gather_rows(f_loc, C),
           "reduce_scatter_d_text_features": lambda: mdist.reduce_scatter_rows(d_full, C),
           "all_reduce_prompt_grads": bucket.all_reduce,  # what the step does: one all-reduce of the flat bucket
           "all_reduce_prompt_grads_rs_ag": lambda: bucket.all_reduce(two_phase=True),
           "all_reduce_loss": lambda: mdist.all_reduce_sum(loss)}
    px = mdist.peer_exchange({}, C, e, device)
    if px is not None:  # the head's exchange as the step does it where the ranks share a node: barrier + own pull kernel
        ops["peer_all_gather_text_features"] = lambda: px.all_gather(0)
        ops["peer_reduce_scatter_d_text_features"] = lambda: px.reduce_scatter(0)
    out = {}
    for name, fn in ops.items():
        for _ in range(3):
            fn()
        dist.barrier()
        torch.cuda.synchronize(device)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize(device)
        t = torch.tensor([e0.elapsed_time(e1) / reps * 1e3], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out[name] = round(float(t), 1)
    return out


def input_pipeline_bench(device, peaks, batch=BATCH_PER_GPU, reps=20):
    """SURVEY 8f N2 beside the headline: the crop / bicubic-resample / flip / normalize kernels on one batch of
    ImageNet-shaped 8-bit images resident in HBM (seeded random crops), CUDA events on the launch stream."""
    import ctypes as C
    import torch
    from mudpt_b200 import _lib
    from mudpt_b200 import input_pipeline as ip
    g = torch.Generator().manual_seed(5)
    shapes = [(375, 500), (500, 375), (333, 500), (480, 640)]
    imgs = [torch.randint(0, 256, (*shapes[i % 4], 3), dtype=torch.uint8, generator=g).to(device) for i in range(batch)]
    tf = ip.GpuTransform(size=(224, 224), is_train=True, device=device)
    torch.manual_seed(5)
    geo = [tf.draw(int(im.shape[0]), int(im.shape[1])) for im in imgs]
    out = tf(imgs, params=geo)  # allocates the workspace, uploads the descriptors
    desc = tf.describe(imgs, geo)
    desc_dev = torch.from_numpy(desc.view("uint8").reshape(-1).copy()).to(device)
    lib = _lib.load()
    host_ptr = desc.ctypes.data_as(C.c_void_p)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)

    def run():
        _lib.check(lib.mudpt_augment_images(desc_dev.data_ptr(), host_ptr, batch, 224, 224, tf.mean, tf.std,
                                            tf._workspace.data_ptr(), tf._workspace.numel(), out.data_ptr(),
                                            _lib.stream_ptr(device)))
    for _ in range(3):
        run()
    ts = []
    for _ in range(reps):
        flush.zero_()  # L2 flush between timed launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); run(); e1.record()
        torch.cuda.synchronize(device)
        ts.append(e0.elapsed_time(e1))
    ms = statistics.median(ts)
    nbytes = sum(int(x[2]) * int(x[3]) * 3 for x in geo) + batch * 3 * 224 * 224 * 4
    return {"kernels": "resample_coeffs_kernel + augment_smem_kernel (bit-exact vs torchvision/PIL bicubic pipeline)",
            "batch": batch, "us_per_batch": round(ms * 1e3, 1), "imgs_per_s": round(batch / (ms * 1e-3), 0),
            "algorithmic_bytes": nbytes, "gbs_algorithmic": round(nbytes / (ms * 1e-3) / 1e9, 1),
            "frac_of_hbm_peak": round(nbytes / (ms * 1e-3) / 1e9 / peaks["hbm"], 4), "l2": "flushed between launches",
            "gpu_launches_per_batch": 2}


def inference_bench(device, batch=256, reps=10):
    """BASELINE configs[2] beside the headline: ViT-B/16 inference with cached text features (1000 classes), batch
    256 per GPU, images resident in HBM (two rotating batches, 308 MB > L2), CUDA events on the launch stream."""
    import torch
    from mudpt_b200 import synthetic as syn
    trainer = build_trainer(device, True)
    model = trainer.model
    imgs = [syn.synthetic_images(batch, 224, seed=200 + i).to(device) for i in range(2)]
    with torch.no_grad():
        model.cache_text_features(device)
        for i in range(3):
            logits = model.inference(imgs[i % 2])
        torch.cuda.synchronize(device)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(reps):
            logits = model.inference(imgs[i % 2])
        e1.record()
        torch.cuda.synchronize(device)
    ms = e0.elapsed_time(e1) / reps
    flops = batch * 35.50e9  # SURVEY.md 8d: vision tower forward, reference formulation
    out = {"workload": "MuDPT ViT-B/16 inference, cached text features, 1000 classes (BASELINE configs[2])", "batch": batch,
           "ms_per_batch": round(ms, 3), "imgs_per_s": round(batch / (ms * 1e-3), 0),
           "tflops_reference_formulation": round(flops / (ms * 1e-3) / 1e12, 1), "finite": bool(torch.isfinite(logits).all())}
    del trainer, model, imgs
    torch.cuda.empty_cache()
    return out

def run_config3(args):
    """BASELINE configs[2] as its own line: inference with cached text features, batch 256 per GPU."""
    import torch
    device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(device)
    r = inference_bench(device, reps=max(args.steps, 5))
    print(json.dumps({"metric": "inference imgs/s MuDPT ViT-B/16 1000-cls, cached text features", "value": r["imgs_per_s"],
                      "unit": UNIT, "n_gpus": 1, "steps": max(args.steps, 5), "warmup": 3, "ms_per_step": r["ms_per_batch"],
                      "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                      "config": {"workload": r["workload"], "batch": r["batch"]}, "detail": r}), flush=True)


def run_config4(args):
    """BASELINE configs[3]: CoCoOp-style instance-conditioned prompts on the shared CLIP kernels -- one train step =
    vision tower (no prompts) -> meta-net -> B x C text sequences in ONE native text-tower pass -> per-image cosine
    logits -> CE -> dgrad through the dense text tower into ctx and the meta-net -> SGD (trainers/cocoop.py:178-198,
    which loops over the images instead).  B = 4 images x 1000 classes per GPU = 4000 sequences of 77 tokens."""
    import torch
    import torch.distributed as dist
    from mudpt_b200 import clip, synthetic as syn
    from mudpt_b200.trainers.cocoop import CustomCLIP
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    B, C = 4, N_CLASSES
    arch = syn.ARCHS["ViT-B/16"]
    cfg = syn.make_cfg(4, 1, "a photo of a", 224, "ViT-B/16")
    cfg.TRAINER["NAME"] = "CoCoOp"
    cfg.TRAINER["COCOOP"] = type(cfg)(N_CTX=4, CTX_INIT="a photo of a", PREC="fp32")
    torch.manual_seed(0)
    clip_model = clip.CLIP(*arch.astuple(), None).float()
    clip_model.load_state_dict(syn.synthetic_clip_state_dict(arch, 0), strict=False)
    model = CustomCLIP(cfg, syn.synthetic_classnames(C), clip_model, tokenizer=syn.synthetic_tokenize)
    for n, p in model.named_parameters():
        if "prompt_learner" not in n:
            p.requires_grad_(False)
    model = model.to(device).train()
    params = [p for p in model.parameters() if p.requires_grad]
    optim = torch.optim.SGD(params, lr=0.002, momentum=0.9, weight_decay=5e-4)
    imgs = [syn.synthetic_images(B, 224, seed=300 + rank * 4 + i).to(device) for i in range(4)]
    labs = [syn.synthetic_labels(B, C, seed=300 + rank * 4 + i).to(device) for i in range(4)]

    def step(i):
        optim.zero_grad(set_to_none=False)
        loss = model(imgs[i % 4], labs[i % 4])
        loss.backward()
        if world > 1:
            from mudpt_b200 import dist as mdist
            mdist.all_reduce_grads(params)
        optim.step()
        return loss

    K, W = max(args.steps, 1), max(args.warmup, 3)
    ms, _, _ = timed_loop(step, K, W, device, world)
    loss = float(step(0))
    if rank == 0:
        eng = clip_model.engine(device)
        print(json.dumps({"metric": "train imgs/s CoCoOp ViT-B/16 1000-cls (B x C text sequences)", "value": B * world / (ms / K * 1e-3),
                          "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True,
                          "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                          "config": {"workload": f"CoCoOp ViT-B/16 train step (BASELINE configs[3]): {B} images x {C} classes per GPU = "
                                                 f"{B * C} text sequences of {eng.text_len} tokens in one text-tower pass, n_ctx 4, "
                                                 "meta-net + ctx trainable, data-parallel over the images",
                                     "text_sequences_per_s": B * C * world / (ms / K * 1e-3)},
                          "loss": loss, "gpu_launches_per_step": None}), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps: exactly K for the train steps of --config 2, 4 and 5; --config 3 times at least 5 "
                         "batches, and --impl reference at most 2 full-size (or 40 sampled) CPU steps so that it ends within "
                         "minutes; the JSON line reports the count used")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--quick", action="store_true", help="profiling aid: resident loop of the full-length variant only")
    ap.add_argument("--classes", type=int, default=N_CLASSES, help="--quick only: classes on this GPU")
    ap.add_argument("--no-overlap", action="store_true", help="--quick only: towers on one stream")
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5],
                    help="BASELINE.json configs (1-based): 2 = the headline (default), 3 = inference with cached text features, "
                         "4 = CoCoOp-shaped step, 5 = ViT-L/14 prompt depth 12")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss, logits, prompt gradients and updated prompt parameters of the last timed train "
                         "step (full-length text tower) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.quick or args.config in (3, 4)):
        ap.error("--dump-outputs applies to the native train step of --config 2 or 5")
    if args.config == 5:
        global ARCH, DEPTH
        ARCH, DEPTH = "ViT-L/14", 12
    # The contract is ONE JSON line on stdout.  Native libraries write there too (NCCL prints its version
    # banner to fd 1 at the first communicator): point fd 1 at stderr for the run and keep the real stdout
    # for the JSON line(s) this script prints itself.
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = real_stdout
    if args.impl == "reference":
        run_reference(args)
    elif args.config == 3:
        run_config3(args)
    elif args.config == 4:
        run_config4(args)
    else:
        run_ours(args)
    real_stdout.flush()


if __name__ == "__main__":
    main()

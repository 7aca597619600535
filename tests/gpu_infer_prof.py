"""Training-forward path against the forward-only (infer) path: time and device memory.

    python tests/gpu_infer_prof.py [--out DIR]   (writes DIR/infer_prof.json)

- config-3 inference (MuDPT ViT-B/16, 1000 classes, cached text features): ms per image batch at B = 256 and 1024;
- device bytes each path holds (mudpt_workspace_bytes);
- the c_fc GEMM at 77,000 x 2048 x 512 (text) and 50,944 x 3072 x 768 (vision, B = 256): modes 3 / 8 against 12 / 13;
- CoCoOp evaluation at 100 images x 1000 classes (infer path only: the training forward would not fit the device).
Medians of >= 10 repetitions, the two paths alternated in the same process; CUDA events around work that ends in a
device synchronise.  Inputs larger than L2 (126 MB) except the c_fc weights.  The card's name, power limit and clocks
are recorded with the numbers.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tests.test_forward_only import _cocoop, _images, _stacks, _vitb16  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.max.sm,clocks.sm,clocks.mem"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return dict(zip(q.split(","), (v.strip() for v in r.stdout.splitlines()[0].split(",")))) if r.returncode == 0 else {}


def timed(fn, reps):
    """ms of each of `reps` calls of fn (each ends in a device synchronise)."""
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1))
    return out


def ab(fns, reps):
    """Alternate the named functions rep by rep; median ms and spread of each."""
    for f in fns.values():  # warm-up (allocation, module load, tensor maps)
        f(); f()
    torch.cuda.synchronize()
    samples = {k: [] for k in fns}
    for _ in range(reps):
        for k, f in fns.items():
            samples[k] += timed(f, 1)
    return {k: {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v), "n": len(v)} for k, v in samples.items()}


def config3(res, reps):
    model = _vitb16(1000)
    eng = model._engine(torch.device("cuda"))
    model.eval()
    with torch.no_grad():
        P_v, P_t = _stacks(model)
        model.cache_text_features()
        f_txt = model._cached_text_features
    for B in (256, 1024):
        img = _images(B, seed=B)
        with torch.no_grad():
            r = ab({"train_forward": lambda: eng.logits_head(eng.vision_forward(img, P_v), f_txt, None, 1.0, False),
                    "infer": lambda: model.inference(img)}, reps)
        r["bytes"] = {p: {t: eng.workspace_bytes(t, k) for t in ("vision", "text")} for p, k in (("train_forward", "train"), ("infer", "infer"))}
        res[f"config3_B{B}"] = r
        print(f"config-3 inference B={B}", json.dumps(r), flush=True)
    del model, eng
    torch.cuda.empty_cache()


def cfc(res, reps):
    from mudpt_b200 import _lib
    from tests.gpu_bringup import _gemm_fused
    lib, st = _lib.load(), _lib.stream_ptr(torch.device("cuda"))
    bf = torch.bfloat16
    for M, N, K in ((77000, 2048, 512), (50944, 3072, 768)):
        torch.manual_seed(0)
        x = torch.randn(M, K, device="cuda")
        xb, stats = torch.empty(M, K, device="cuda", dtype=bf), torch.empty(M, K // 64, 2, device="cuda")
        _lib.check(lib.mudpt_rowstats(x.data_ptr(), xb.data_ptr(), stats.data_ptr(), M, K, st))
        W = (torch.randn(N, K, device="cuda") * K ** -0.5).to(bf)
        bias, cs = torch.randn(N, device="cuda"), torch.randn(N, device="cuda")
        h, g = torch.empty(M, N, device="cuda", dtype=bf), torch.empty(M, N, device="cuda", dtype=bf)
        ln = dict(bias=bias, colsum=cs, ln_stats=stats, ln_parts=K // 64, ln_width=K)
        n = 20  # launches per sample

        def run(mode, **kw):
            def f():
                for _ in range(n):
                    _gemm_fused(lib, st, xb, W, M, N, K, mode=mode, stream_k=-1, **kw)
            return f
        r = ab({"m3": run(3, out0=h, out1=g, bias=bias), "m12": run(12, out0=g, bias=bias),
                "m8": run(8, out0=h, out1=g, **ln), "m13": run(13, out0=g, **ln)}, reps)
        for v in r.values():
            v["us_per_launch"] = 1e3 * v["median_ms"] / n
        r["write_bytes"] = {"m3_m8": 2 * 2 * M * N, "m12_m13": 2 * M * N}
        r["mma_bound_us"] = 2.0 * M * N * K / 2.25e15 * 1e6  # data-sheet dense BF16 rate, not a measured figure
        res[f"cfc_{M}x{N}x{K}"] = r
        print(f"c_fc {M}x{N}x{K}", json.dumps(r), flush=True)
        del x, xb, stats, h, g
        torch.cuda.empty_cache()


def cocoop_eval(res, reps):
    model = _cocoop(1000)
    eng = model._clip_ref[0].engine()
    model.eval()
    img = _images(100, seed=3)
    with torch.no_grad():
        r = ab({"infer": lambda: model(img)}, reps)
    r["rows"] = eng.n_classes * eng.text_len
    r["bytes"] = {"text_infer": eng.workspace_bytes("text", "infer"), "text_input": eng.workspace_bytes("text", "input"),
                  "text_train": eng.workspace_bytes("text", "train")}
    r["peak_allocated_torch"] = torch.cuda.max_memory_allocated()
    res["cocoop_eval_100x1000"] = r
    print("CoCoOp eval 100 x 1000", json.dumps(r), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.environ.get("TMPDIR", "/tmp"), "mudpt_infer_prof"))
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    res = {"gpu": gpu_info()}
    print(res["gpu"], flush=True)
    config3(res, a.reps)
    cfc(res, a.reps)
    cocoop_eval(res, a.reps)
    res["gpu_after"] = gpu_info()
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "infer_prof.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

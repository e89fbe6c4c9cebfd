#!/usr/bin/env python
"""difference_score_function (S = 1 / |p - z|^2): fused InfoNCE kernels against the literal path, on the device.

    python tools/profile_difference_score.py [--out profiles/difference_score.json] [--iters 50]

At (B, K, E) = (64, 16, 256) (experiments e4 / e5), lambda = 0.01, both modes: forward + backward time (CUDA events
over --iters calls after warm-up) and peak torch.cuda.max_memory_allocated of the fused path and of the literal one
(trainer.difference_score_function + reference_loss_from_scores + backward).  Then all-steps batch scaling,
B = 64 ... 1024: the fused path at every size; the literal path only while its peak, predicted from the peak measured at
the previous size times (B / B_prev)^2, stays below half of the free device memory -- the GPU may be shared, so an
allocation expected to fail is never attempted.  Prints one JSON line and writes it to --out.
"""
import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "constrastive-predictive-coding-audio_b200"))
import torch                                                    # noqa: E402
import cpc_b200                                                 # noqa: E402
from cpc_b200 import trainer as T                               # noqa: E402

DEV = torch.device("cuda:0")
REG = 0.01


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (v.strip() for v in out.split(","))
    return name, power


def inputs(b, k, e):
    g = torch.Generator(device=DEV).manual_seed(b + k + e)
    pred = (torch.randn(b, k, e, generator=g, device=DEV) / math.sqrt(e)).requires_grad_(True)
    z = (torch.randn(b, e, k, generator=g, device=DEV) / math.sqrt(e)).requires_grad_(True)
    return pred, z


def fused_step(pred, z, all_steps):
    pred.grad = z.grad = None
    loss = cpc_b200.ops.infonce(pred, z, all_steps, "difference", REG)[0]
    loss.backward()
    return loss


def literal_step(pred, z, all_steps):
    pred.grad = z.grad = None
    b, k, _ = pred.shape
    loss, _ = T.reference_loss_from_scores(T.difference_score_function(pred, z), b, k, all_steps, REG)
    loss.backward()
    return loss


def measure(step, pred, z, all_steps, iters):
    """(ms per forward + backward, peak MB of one call, loss)"""
    for _ in range(3):
        loss = step(pred, z, all_steps)
    torch.cuda.synchronize()
    pred.grad = z.grad = None
    torch.cuda.reset_peak_memory_stats(DEV)
    loss = step(pred, z, all_steps)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated(DEV) / 2 ** 20
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(iters):
        step(pred, z, all_steps)
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / iters, peak, float(loss)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "difference_score.json"))
    ap.add_argument("--iters", type=int, default=50)
    args = ap.parse_args()
    if args.iters < 1:
        raise SystemExit("--iters must be >= 1")
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures on the GPU only")
    name, power = card()
    b, k, e = 64, 16, 256
    res = {"tool": "tools/profile_difference_score.py", "gpu": name, "power_limit": power, "torch": torch.__version__,
           "shape_bke": [b, k, e], "regularization": REG, "iters": args.iters, "modes": {}, "batch_scaling_all_steps": []}
    for all_steps in (True, False):
        pred, z = inputs(b, k, e)
        f_ms, f_mb, f_loss = measure(fused_step, pred, z, all_steps, args.iters)
        l_ms, l_mb, l_loss = measure(literal_step, pred, z, all_steps, args.iters)
        res["modes"]["all_steps" if all_steps else "per_step"] = {
            "fused_ms": round(f_ms, 4), "literal_ms": round(l_ms, 4), "speedup": round(l_ms / f_ms, 2),
            "fused_peak_mb": round(f_mb, 1), "literal_peak_mb": round(l_mb, 1),
            "loss_fused": f_loss, "loss_literal": l_loss}
        del pred, z
        torch.cuda.empty_cache()
    prev = None                                                  # (batch, literal peak bytes) of the last literal run
    for bs in (64, 128, 256, 512, 1024):
        pred, z = inputs(bs, k, e)
        f_ms, f_mb, _ = measure(fused_step, pred, z, True, args.iters)
        row = {"batch": bs, "candidates": bs * k, "fused_ms": round(f_ms, 4), "fused_peak_mb": round(f_mb, 1)}
        free = torch.cuda.mem_get_info(DEV)[0]
        predicted = None if prev is None else prev[1] * (bs / prev[0]) ** 2
        if predicted is not None and predicted >= free / 2:
            row["literal"] = "not run (predicted %.1f GB)" % (predicted / 1e9)
            prev = (bs, predicted)                               # later sizes are predicted from this one
        else:
            l_ms, l_mb, _ = measure(literal_step, pred, z, True, args.iters)
            row.update(literal_ms=round(l_ms, 4), literal_peak_mb=round(l_mb, 1), speedup=round(l_ms / f_ms, 2))
            prev = (bs, l_mb * 2 ** 20)
        row["free_gb_before_literal"] = round(free / 1e9, 1)
        res["batch_scaling_all_steps"].append(row)
        del pred, z
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write(line + "\n")


if __name__ == "__main__":
    main()

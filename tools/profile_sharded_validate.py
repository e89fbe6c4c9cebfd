#!/usr/bin/env python
"""Sharded validation: what one rank spends on one validation batch of e24, on one device.

    python tools/profile_sharded_validate.py [--out profiles/sharded_validate.json] [--iters 10] [--reps 5]

For W = 1, 2, 4, 8 and the reference's validation batch of 64 items, two eager paths (model in eval mode, no autograd):
  "full"  -- what every rank does in validate(): forward of all 64 items, then the square metrics kernel
             (ops.infonce_validate);
  "shard" -- what rank W-1 does in validate(shard_over_ranks=True): forward of its b = 64/W items, the rectangular
             metrics of its targets against 64 gathered predictions (ops.infonce_validate_shard) and the combine of W
             records (ops.infonce_validate_combine).
The collectives are not part of either: on one device the gathered predictions are W copies of the shard's and the W
records are copies of its own, so the times leave out the two all-gathers (a few hundred kB) a real run adds.  The
metrics calls alone are timed as well ("metrics_full", "metrics_shard").  CUDA events around --iters calls, the paths
alternated --reps times, medians reported.  Prints one JSON line with the card name and power limit and writes it to
--out.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "constrastive-predictive-coding-audio_b200"))
import torch                                                    # noqa: E402
import cpc_b200                                                 # noqa: E402

BATCH = 64


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (v.strip() for v in out.split(","))
    return name, power


def events_ms(fn, iters):
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(iters):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "sharded_validate.json"))
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if args.iters < 1 or args.reps < 1:
        raise SystemExit("--iters and --reps must be >= 1")
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures on the GPU only")
    dev = torch.device("cuda", 0)
    name, power = card()
    exp = cpc_b200.configs.experiment("e24")
    tc = exp["training_config"]
    all_steps, k = tc["score_over_all_timesteps"], tc["prediction_steps"]
    kind = cpc_b200.trainer._FUSED_KINDS[tc["score_function"]]
    torch.manual_seed(0)
    model, pre, _ = cpc_b200.configs.setup_model(exp["cqt_config"], exp["encoder_config"], exp["ar_model_config"], tc,
                                                 device=dev)
    model.eval()
    audio = (0.1 * torch.randn(BATCH, model.item_length, generator=torch.Generator().manual_seed(7))).to(dev)

    def forward(x):
        x = x.unsqueeze(1)
        if pre is not None:
            x = pre(x)
        return model(x)[:2]

    rows = []
    with torch.no_grad():
        pred_full, tgt_full = forward(audio)
        for world in (1, 2, 4, 8):
            b = BATCH // world
            shard = audio[(world - 1) * b:]
            pred_s, tgt_s = forward(shard)
            pred_all = pred_s.repeat(world, 1, 1)                   # stands in for the all-gather

            def metrics_full():
                return cpc_b200.ops.infonce_validate(pred_full, tgt_full, all_steps, kind)

            def metrics_shard():
                rec = cpc_b200.ops.infonce_validate_shard(pred_all, tgt_s, all_steps, kind, (world - 1) * b)
                return cpc_b200.ops.infonce_validate_combine(rec.unsqueeze(0).expand(world, -1), b, k, all_steps)

            def full():
                p, t = forward(audio)
                return cpc_b200.ops.infonce_validate(p, t, all_steps, kind)

            def sharded():
                p, t = forward(shard)
                rec = cpc_b200.ops.infonce_validate_shard(p.repeat(world, 1, 1), t, all_steps, kind, (world - 1) * b)
                return cpc_b200.ops.infonce_validate_combine(rec.unsqueeze(0).expand(world, -1), b, k, all_steps)

            paths = {"full": full, "shard": sharded, "metrics_full": metrics_full, "metrics_shard": metrics_shard}
            for fn in paths.values():                               # warm-up of every shape
                fn()
            torch.cuda.synchronize()
            times = {n: [] for n in paths}
            for _ in range(args.reps):
                for n, fn in paths.items():
                    times[n].append(events_ms(fn, args.iters))
            med = {n: statistics.median(v) for n, v in times.items()}
            rows.append({"world": world, "shard_items": b, **{n + "_ms": round(v, 4) for n, v in med.items()},
                         "shard_over_full": round(med["shard"] / med["full"], 3), "ideal": round(1.0 / world, 3),
                         "ms_all": {n: [round(x, 4) for x in v] for n, v in times.items()}})
    res = {"tool": "tools/profile_sharded_validate.py", "gpu": name, "power_limit": power, "torch": torch.__version__,
           "workload": "e24 validation batch of %d items (K = %d, %s, %s), eval mode" % (
               BATCH, k, "all-steps" if all_steps else "per-step", kind),
           "timing": "eager, CUDA events over iters calls, median of reps; collectives not included",
           "iters": args.iters, "reps": args.reps, "rows": rows}
    line = json.dumps(res)
    print(line, flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write(line + "\n")


if __name__ == "__main__":
    main()

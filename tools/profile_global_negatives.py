#!/usr/bin/env python
"""Global negatives: cost of the rectangular (shard) InfoNCE call and of the option in e24's training step, on the device.

    python tools/profile_global_negatives.py [--out profiles/global_negatives.json] [--iters 50] [--reps 5]
    python -m torch.distributed.run --nproc-per-node N tools/profile_global_negatives.py --step [--iters 20]

(a) one GPU (default): at e24's shard shape (b = 64, K = 16, E = 512, linear, all-steps, lambda = 0), in the fp32 and
    the bf16 operand modes, forward + backward of the rectangular call (predictions of W*b items, this shard's b
    targets) for W = 1, 2, 4, 8, next to the square call over N = W*b items.  Each call is captured --iters times into a
    CUDA graph after a warm-up, so a replay timed with CUDA events is device time, free of the host's submission cost;
    the two graphs alternate --reps times and the median of each is reported.  The rectangle does 1/W of the square's
    work.
(b) --step, under torch.distributed.run: ms per e24 GraphedTrainStep (b = 64 per GPU) with per-GPU and with global
    negatives, alternated --reps times, median of the slowest rank.
Prints one JSON line with the card name and power limit and writes it to --out (rank 0).
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "constrastive-predictive-coding-audio_b200"))
import torch                                                    # noqa: E402
import cpc_b200                                                 # noqa: E402

B, K, E = 64, 16, 512


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


def graphed(fn, iters):
    """fn() warmed up on a side stream, then captured iters times into one CUDA graph."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(iters):
            fn()
    torch.cuda.synchronize()
    return graph


def kernel_calls(args, dev):
    rows = []
    for precision in ("fp32", "bf16"):
        for world in (1, 2, 4, 8):
            n = world * B
            g = torch.Generator(device=dev).manual_seed(world)
            pred = (torch.randn(n, K, E, generator=g, device=dev) / math.sqrt(E)).requires_grad_(True)
            z = (torch.randn(n, E, K + 4, generator=g, device=dev) / math.sqrt(E)).requires_grad_(True)
            off = (world - 1) * B                                          # the last rank's shard

            def rect():
                pred.grad = z.grad = None
                cpc_b200.ops.infonce(pred, z[off:off + B, :, -K:], True, "linear", 0.0, precision=precision,
                                     target_offset=off)[0].backward()

            def square():
                pred.grad = z.grad = None
                cpc_b200.ops.infonce(pred, z[:, :, -K:], True, "linear", 0.0, precision=precision)[0].backward()

            g_rect, g_square = graphed(rect, args.iters), graphed(square, args.iters)
            r_ms, s_ms = [], []
            for _ in range(args.reps):
                r_ms.append(events_ms(g_rect.replay, 1) / args.iters)
                s_ms.append(events_ms(g_square.replay, 1) / args.iters)
            r, s = statistics.median(r_ms), statistics.median(s_ms)
            rows.append({"precision": precision, "world": world, "rect_ms": round(r, 4), "square_ms": round(s, 4),
                         "rect_over_square": round(r / s, 3), "ideal": round(1.0 / world, 3),
                         "rect_ms_all": [round(v, 4) for v in r_ms], "square_ms_all": [round(v, 4) for v in s_ms]})
            del pred, z, g_rect, g_square
            torch.cuda.empty_cache()
    return {"shape_bke": [B, K, E], "mode": "all-steps linear, lambda 0", "timing": "CUDA graph of iters calls",
            "iters": args.iters, "reps": args.reps, "rows": rows}


def train_steps(args, dev, rank, world):
    import torch.distributed as dist
    from cpc_b200 import configs, ddp
    exp = configs.experiment("e24")
    tc = exp["training_config"]
    steps = {}
    for flag in (False, True):
        torch.manual_seed(0)
        model, pre, _ = configs.setup_model(exp["cqt_config"], exp["encoder_config"], exp["ar_model_config"], tc,
                                            device=dev)
        ddp.broadcast_parameters(model, 0)
        trainer = cpc_b200.ContrastiveEstimationTrainer(
            model=model, dataset=None, device=dev, regularization=tc["regularization"],
            score_over_all_timesteps=tc["score_over_all_timesteps"], score_function=tc["score_function"],
            preprocessing=pre, prediction_steps=tc["prediction_steps"], verbose=False, global_negatives=flag)
        model.train()
        step = cpc_b200.GraphedTrainStep(trainer, trainer.make_optimizer(tc["learning_rate"]), (B, model.item_length))
        steps["global" if flag else "per_gpu"] = (step, model.item_length)
    g = torch.Generator().manual_seed(1234 + rank)
    batch = (0.1 * torch.randn(B, steps["per_gpu"][1], generator=g)).to(dev)
    times = {name: [] for name in steps}
    losses = {}
    for _ in range(args.reps):
        for name, (step, _) in steps.items():
            for _ in range(2):
                step(batch)
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            ms = events_ms(lambda: step(batch), args.iters)
            t = torch.tensor([ms], device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            times[name].append(t.item())
            losses[name] = step.loss.item()
    return {"workload": "e24 GraphedTrainStep, b = %d per GPU" % B, "world": world, "iters": args.iters,
            "reps": args.reps, "ms_per_step": {n: round(statistics.median(v), 3) for n, v in times.items()},
            "ms_all": {n: [round(x, 3) for x in v] for n, v in times.items()}, "last_loss": losses}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "global_negatives.json"))
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--step", action="store_true", help="(b): e24 training steps under torch.distributed.run")
    args = ap.parse_args()
    if args.iters < 1 or args.reps < 1:
        raise SystemExit("--iters and --reps must be >= 1")
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures on the GPU only")
    from cpc_b200 import ddp
    rank, world, local = ddp.init_from_env("nccl") if args.step else (0, 1, 0)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    name, power = card()
    res = {"tool": "tools/profile_global_negatives.py", "gpu": name, "power_limit": power, "torch": torch.__version__}
    if args.step:
        res["train_step"] = train_steps(args, dev, rank, world)
    else:
        res["kernel_calls"] = kernel_calls(args, dev)
    if rank == 0:
        line = json.dumps(res)
        print(line, flush=True)
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        os._exit(0)                                              # skip interpreter teardown of graphs holding NCCL work


if __name__ == "__main__":
    main()

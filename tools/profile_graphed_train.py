#!/usr/bin/env python
"""What ``train(cuda_graph=True)`` saves over the eager loop: e24 at B = 64, fed from WAV files by the device loader.

    python tools/profile_graphed_train.py [--out FILE] [--steps 10] [--warmup 3] [--reps 3]

Writes a synthetic folder of 16-bit mono WAV files (e24 items of 97 024 samples) under a temporary directory, as
tools/profile_device_loader.py does, then alternates ``train(device_loading=True)`` and
``train(device_loading=True, cuda_graph=True)`` --reps times each.  Every step ends in the loop's host read of the
loss, so a host clock between the logger calls of two steps is the step's wall time: ms per step is the clock over
--steps steps after --warmup steps, and the reported value is the median over the repetitions.  The graph's capture
(``GraphedTrainStep`` construction, warm-up steps included) is timed once per graphed run as a one-off cost.  Prints
one JSON line with the card name and power limit, and also writes it to --out when given (profiles/graphed_train.json
holds the line DESIGN.md §6.1 quotes).
"""
import argparse
import json
import os
import random
import statistics
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "constrastive-predictive-coding-audio_b200"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch                                                    # noqa: E402
import cpc_b200                                                 # noqa: E402
from cpc_b200 import trainer as T                               # noqa: E402
from profile_device_loader import BATCH, ITEM, card, write_folder   # noqa: E402


class _Meter:
    def update(self, value):
        pass


class StampLogger:
    """train()'s per-step logger interface; records the host clock at each step's log call."""

    def __init__(self):
        self.loss_meter, self.score_meter, self.stamps = _Meter(), _Meter(), []

    def log(self, step):
        self.stamps.append(time.perf_counter())


class TimedGraphedTrainStep(T.GraphedTrainStep):
    captures = []

    def __init__(self, *args, **kwargs):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        super().__init__(*args, **kwargs)
        torch.cuda.synchronize()
        self.captures.append((time.perf_counter() - t0) * 1e3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script times GPU steps")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"tool": "tools/profile_graphed_train.py", "torch": torch.__version__, "batch": BATCH, "item_length": ITEM,
           "steps": args.steps, "warmup": args.warmup, "reps": args.reps}
    res["gpu"], res["power_limit"] = card()
    T.GraphedTrainStep = TimedGraphedTrainStep                  # train() builds its graph through this name
    exp = cpc_b200.configs.experiment("e24")
    tc = exp["training_config"]
    torch.manual_seed(0)
    model, pre, _ = cpc_b200.configs.setup_model(exp["cqt_config"], exp["encoder_config"], exp["ar_model_config"], tc,
                                                 device=dev)
    assert model.item_length == ITEM, model.item_length
    per_file = 24
    n_steps = args.warmup + args.steps
    with tempfile.TemporaryDirectory() as tmp:
        ds = write_folder(os.path.join(tmp, "m16"), -(-BATCH * (n_steps + 2) // per_file), per_file * ITEM + 1000, 1, 2, 1)
        logger = StampLogger()
        trainer = cpc_b200.ContrastiveEstimationTrainer(model=model, dataset=ds, device=dev, preprocessing=pre,
                                                        logger=logger,
                                                        score_over_all_timesteps=tc["score_over_all_timesteps"],
                                                        score_function=tc["score_function"],
                                                        prediction_steps=tc["prediction_steps"], verbose=False)
        runs = {"eager": [], "cuda_graph": []}
        for _ in range(args.reps):
            for name, graph in (("eager", False), ("cuda_graph", True)):
                logger.stamps.clear()
                random.seed(0)
                trainer.train(batch_size=BATCH, epochs=1, lr=1e-4, max_steps=n_steps, device_loading=True,
                              cuda_graph=graph)
                assert len(logger.stamps) == n_steps, len(logger.stamps)
                s = logger.stamps
                runs[name].append(round((s[n_steps - 1] - s[args.warmup - 1]) * 1e3 / args.steps, 3))
    res["e24_train_device_loading_ms_per_step"] = {k: {"median": statistics.median(v), "runs": v}
                                                   for k, v in runs.items()}
    res["capture_ms"] = {"median": round(statistics.median(TimedGraphedTrainStep.captures), 1),
                         "runs": [round(c, 1) for c in TimedGraphedTrainStep.captures]}
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()

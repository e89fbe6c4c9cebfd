#!/usr/bin/env python
"""What it costs to feed e24 training from WAV files: the DataLoader path against DeviceBatchLoader.

    python tools/profile_device_loader.py [--out FILE] [--batches 6] [--steps 10] [--host-only]

Writes synthetic WAV folders under a temporary directory: e24 items (97 024 samples) of 16-bit mono audio, and the
same of 24-bit stereo audio.  Then, for 64-item batches:
  host (any machine) -- ms per batch of ``DataLoader(AudioDataset, num_workers=0/1/4)`` (wall time per batch
      delivered; with 0 workers that is the consuming core's CPU time), and the device loader's producer work per batch
      (``SegmentPlanner.stage``: planning + memmap copies, wall and thread CPU time);
  GPU (skipped with --host-only) -- kernel time of ``ops.pcm_assemble`` (CUDA events over 50 calls, batch resident on
      the device), upload time of one staged batch from pinned memory (CUDA events over 20 copies), and eager e24
      ``train()`` ms per step from the 16-bit files with ``num_workers=4``, with ``device_loading=True``, and the same
      step body fed from one resident device batch.
Prints one JSON line with the card name, power limit and host core count, and also writes it to --out when given
(profiles/device_loader.json holds the line DESIGN.md §6.1 quotes).
"""
import argparse
import json
import os
import random
import subprocess
import sys
import tempfile
import time
import wave

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "constrastive-predictive-coding-audio_b200"))
import torch                                                    # noqa: E402
import cpc_b200                                                 # noqa: E402
from cpc_b200.audio_dataset import AudioDataset                 # noqa: E402
from cpc_b200.device_loader import DeviceBatchLoader, SegmentPlanner  # noqa: E402
from cpc_b200.sampler import FileBatchSampler                   # noqa: E402

BATCH, ITEM = 64, 97024


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    return [v.strip() for v in out.split(",")]


def write_folder(root, n_files, frames, channels, width, seed):
    os.makedirs(root)
    rng = np.random.default_rng(seed)
    for i in range(n_files):
        x = (rng.standard_normal((frames, channels)) * 0.1 * (1 << (8 * width - 1))).astype(np.int64)
        if width == 3:
            v = x & 0xFFFFFF
            raw = np.stack([v & 0xFF, (v >> 8) & 0xFF, (v >> 16) & 0xFF], axis=-1).astype(np.uint8).tobytes()
        else:
            raw = x.astype("<i2").tobytes()
        with wave.open(os.path.join(root, "f%02d.wav" % i), "wb") as fh:
            fh.setnchannels(channels)
            fh.setsampwidth(width)
            fh.setframerate(16000)
            fh.writeframes(raw)
    return AudioDataset(root, item_length=ITEM, unique_length=ITEM)


def batches_of(ds, n):
    random.seed(0)
    sampler = FileBatchSampler(ds.get_example_count_per_file(), batch_size=BATCH, drop_last=True)
    out = list(sampler)[:n]
    assert len(out) == n, "dataset too small for %d batches" % n
    return out


def dataloader_ms(ds, batches, workers, pin):
    loader = torch.utils.data.DataLoader(ds, batch_sampler=batches, num_workers=workers, pin_memory=pin)
    it = iter(loader)
    next(it)                                                    # worker start-up is not part of the rate
    t0 = time.perf_counter()
    n = sum(1 for _ in it)
    ms = (time.perf_counter() - t0) * 1e3 / n
    del it, loader
    return round(ms, 2)


def stage_ms(planner, batches):
    holder = {}

    def buffer_for(nbytes):
        if holder.get("buf") is None or holder["buf"].size < nbytes:
            holder["buf"] = np.empty(nbytes, dtype=np.uint8)
        return holder["buf"]
    planner.stage(batches[0], buffer_for)                       # maps opened, buffer faulted in
    t0, c0 = time.perf_counter(), time.thread_time()
    for b in batches[1:]:
        planner.stage(b, buffer_for)
    n = len(batches) - 1
    return round((time.perf_counter() - t0) * 1e3 / n, 3), round((time.thread_time() - c0) * 1e3 / n, 3)


def host_rows(datasets, batches_n, pin):
    rows = {}
    for name, ds in datasets.items():
        batches = batches_of(ds, batches_n)
        row = {"dataloader_ms_per_batch": {str(w): dataloader_ms(ds, batches, w, pin) for w in (0, 1, 4)}}
        wall, cpu = stage_ms(SegmentPlanner(ds), batches)
        row["producer_stage_ms_per_batch"] = {"wall": wall, "thread_cpu": cpu}
        rows[name] = row
    return rows


def events_ms(fn, iters):
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(iters):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / iters


def kernel_rows(datasets, dev):
    rows = {}
    for name, ds in datasets.items():
        planner = SegmentPlanner(ds)
        batch = batches_of(ds, 1)[0]
        host = {}
        table, header, total = planner.stage(batch, lambda n: host.setdefault(
            "t", torch.empty(n, dtype=torch.uint8, pin_memory=True)).numpy())
        pinned = host["t"]
        staged = pinned.to(dev)
        out = torch.empty(BATCH, ITEM, device=dev)

        def kernel():
            cpc_b200.ops.pcm_assemble(table, staged[:table.nbytes], staged[header:total], out)

        def upload():
            staged.copy_(pinned, non_blocking=True)
        kernel(), upload()
        torch.cuda.synchronize()
        assert torch.equal(out.cpu(), torch.stack([ds[i] for i in batch]))
        k_ms = min(events_ms(kernel, 50) for _ in range(3))
        u_ms = min(events_ms(upload, 20) for _ in range(3))
        rows[name] = {"kernel_us": round(k_ms * 1e3, 2), "upload_ms": round(u_ms, 3), "staged_bytes": int(total),
                      "kernel_GBps": round((total - header + 4 * BATCH * ITEM) / (k_ms * 1e-3) / 1e9, 1),
                      "upload_GBps": round(total / (u_ms * 1e-3) / 1e9, 1)}
    return rows


def train_rows(ds, dev, steps, warm=3):
    exp = cpc_b200.configs.experiment("e24")
    tc = exp["training_config"]
    torch.manual_seed(0)
    model, pre, _ = cpc_b200.configs.setup_model(exp["cqt_config"], exp["encoder_config"], exp["ar_model_config"], tc,
                                                 device=dev)
    assert model.item_length == ITEM, model.item_length
    trainer = cpc_b200.ContrastiveEstimationTrainer(model=model, dataset=ds, device=dev, preprocessing=pre,
                                                    score_over_all_timesteps=tc["score_over_all_timesteps"],
                                                    score_function=tc["score_function"],
                                                    prediction_steps=tc["prediction_steps"], verbose=False)
    plain = trainer.loss_on_batch
    stamps = []

    def stamped(batch):
        stamps.append(time.perf_counter())
        return plain(batch)
    trainer.loss_on_batch = stamped
    rows = {}
    for name, kw in (("dataloader_4_workers", dict(num_workers=4)), ("device_loading", dict(device_loading=True))):
        stamps.clear()
        random.seed(0)
        trainer.train(batch_size=BATCH, epochs=1, lr=1e-4, max_steps=warm + steps + 1, **kw)
        rows[name] = round((stamps[warm + steps] - stamps[warm]) * 1e3 / steps, 2)
    # the same step body (train()'s loop) on one resident batch
    trainer.loss_on_batch = plain
    optimizer = trainer.make_optimizer(1e-4)
    resident = torch.stack([ds[i] for i in batches_of(ds, 1)[0]]).to(dev)
    for i in range(warm + steps):
        if i == warm:
            t0 = time.perf_counter()
        loss, mx = trainer.loss_on_batch(resident)
        assert not trainer._any_rank_nan(loss)
        trainer.model.zero_grad()
        loss.backward()
        optimizer.step()
        torch.stack([loss.detach(), mx.detach()]).tolist()
    rows["resident_batch"] = round((time.perf_counter() - t0) * 1e3 / steps, 2)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    ap.add_argument("--batches", type=int, default=6)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--host-only", action="store_true")
    args = ap.parse_args()
    if not args.host_only and not torch.cuda.is_available():
        raise SystemExit("no CUDA device: run with --host-only for the host part")
    res = {"tool": "tools/profile_device_loader.py", "torch": torch.__version__, "host_cores": os.cpu_count(),
           "usable_cores": len(os.sched_getaffinity(0)), "batch": BATCH, "item_length": ITEM}
    if not args.host_only:
        res["gpu"], res["power_limit"] = card()
    train_items = BATCH * (args.steps + 5)
    per_file = 24                                               # items per file; 1000 spare frames cover the crossings
    with tempfile.TemporaryDirectory() as tmp:
        datasets = {
            "16bit_mono": write_folder(os.path.join(tmp, "m16"), -(-train_items // per_file), per_file * ITEM + 1000, 1, 2, 1),
            "24bit_stereo": write_folder(os.path.join(tmp, "s24"), -(-BATCH * args.batches // per_file) + 1,
                                         per_file * ITEM + 1000, 2, 3, 2)}
        res["host"] = host_rows(datasets, args.batches, pin=not args.host_only)
        if not args.host_only:
            dev = torch.device("cuda", 0)
            torch.cuda.set_device(dev)
            res["gpu_kernel"] = kernel_rows(datasets, dev)
            res["e24_train_ms_per_step_16bit_mono"] = train_rows(datasets["16bit_mono"], dev, args.steps)
    res["not_measured"] = "wall clock of 8 ranks feeding 8 GPUs (one GPU here)"
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()

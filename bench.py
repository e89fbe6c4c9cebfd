#!/usr/bin/env python
"""bench.py -- train audio-sec/sec of the CPC hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload NAME] [--batch B]
                    [--dump-outputs DIR]

Workloads (``--workload``; the default is the one BASELINE.json's metric is quoted on):

  e24          BASELINE configs[1] = experiments['e24'] of the reference: CQT(+phase) PreprocessingModule ->
               ScalogramResidualEncoder arch 7 -> ConvolutionalArModel arch 3 -> InfoNCE (linear, all-steps, K=16),
               batch 64 items of 97 024 samples (6.064 s at 16 kHz) PER GPU (weak scaling), Adam step included.
  raw_wave     BASELINE configs[0]: AudioEncoder (512 ch) + AudioGRUModel(512, 256), K=12, V=100, softplus per-step
               scoring with regulariser 1 (the trainer's defaults), items of 18 385 samples, batch 8 per GPU.
  e20_bf16     BASELINE configs[2]: arch 7 + AttentionModel (attention_architecture_1), bf16 operand mode of the conv
               kernels (fp32 accumulate, fp32 batch norm / loss), batch 64 per GPU.
  long_context BASELINE configs[4]: the e24 model with visible_steps=112 (items of 150 272 samples = 9.39 s, 1046 CQT
               frames), batch 64 per GPU.
  e29          the reference's default experiment (high-res CQT, arch 9, attention AR, gradient penalty), batch 16, eager.
  infonce_sweep BASELINE configs[3]: the fused InfoNCE forward + backward alone over candidates 128...8192 x K 4...32.

One "step" = one full training step (CQT -> encoder -> AR -> InfoNCE forward/backward -> Adam) on synthetic white-noise
audio with random-init weights.  Our arm prints `value` (inputs resident in HBM), `e2e` (the same step through the public
trainer objects with every batch coming from pinned host memory and the loss read back every step), `roofline` of the
single most expensive kernel (one entry point at one shape, timed with CUDA events inside real steps), `metrics`
(CQT GB/s and dense-equivalent TFLOP/s, InfoNCE TFLOP/s, conv TFLOP/s by kernel family) and `cpu_baseline` (the oracle
port of the same step on the host cores, bounded sample).  `--impl reference` times that CPU port alone (the reference is
CPU-only Python, so kind = "port").

`--dump-outputs DIR` writes what the last timed step computed (rank 0) as float32 .npy files: loss.npy and max_score.npy
(what the step returns) and gradients.npy (the gradient of every trainable parameter that the optimizer applies, i.e.
averaged over ranks, flattened and concatenated in model.parameters() order). An array longer than DUMP_SAMPLE entries
is stored as a fixed, seeded sample of DUMP_SAMPLE entries (in index order). Every timed step starts from the seeded
initial state (see run_ours) on seeded batches, so two runs, or two builds, run with the same arguments can be compared
output for output: one run of a build repeats another up to the rounding of a single step. Each timed step is timed
alone with its own CUDA events, so the restore before it and any gap between steps are not timed, and each is the
optimizer's first step. The parameters after the optimizer step are not written: a conv bias that feeds a train-mode
batch norm has a true gradient of exactly zero, so its computed gradient is rounding noise, and Adam turns that noise
into a step of +-lr.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "constrastive-predictive-coding-audio_b200")
sys.path.insert(0, PKG)

SR = 16000
METRIC = "train audio-sec/sec"
DUMP_SAMPLE = 1 << 22                                           # entries kept of a longer dumped array (16 MB in fp32)

WORKLOADS = {
    "e24": {"batch": 64, "cpu_batch": 8, "visible": 60, "prediction": 16, "dtype": "f32",
            "text": "e24: CQT(256 bins, phase) + ScalogramResidualEncoder arch7 + ConvolutionalArModel arch3 + InfoNCE "
                    "linear/all-steps K=16, full train step incl. Adam (BASELINE configs[1])"},
    "raw_wave": {"batch": 8, "cpu_batch": 8, "visible": 100, "prediction": 12, "dtype": "f32",
                 "text": "raw_wave: AudioEncoder 512ch (strides 5,4,2,2,2) + AudioGRUModel(512,256) + InfoNCE softplus/"
                         "per-step K=12 reg=1, full train step incl. Adam (BASELINE configs[0])"},
    "e20_bf16": {"batch": 64, "cpu_batch": None, "visible": 60, "prediction": 16, "dtype": "bf16",
                 "text": "e20_bf16: CQT(256 bins, phase) + ScalogramResidualEncoder arch7 + AttentionModel "
                         "(attention_architecture_1) + InfoNCE linear/all-steps K=16, conv kernels in bf16-operand mode, "
                         "full train step incl. Adam (BASELINE configs[2])"},
    "e29": {"batch": 16, "cpu_batch": None, "visible": 43, "prediction": 16, "dtype": "f32", "sr": 44100, "graph": False,
            "text": "e29 (the reference's default experiment, train_script.py:11): high-res CQT (44.1 kHz, 292 bins, hop 256) + "
                    "offset/pooled scalogram + resnet arch 9 + AttentionModel + InfoNCE linear/all-steps K=16 with the "
                    "Wasserstein gradient penalty (second-order autograd), batch 16 as configured, eager submission"},
    "long_context": {"batch": 64, "cpu_batch": 4, "visible": 112, "prediction": 16, "dtype": "f32",
                     "text": "long_context: the e24 model with visible_steps=112: items of 150 272 samples (9.39 s, 1046 "
                             "CQT frames x 256 bins), full train step incl. Adam (BASELINE configs[4])"},
}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        return {"hbm": p["hbm_gbs"], "tensor_burst": p["bf16_tflops"], "tensor": p["bf16_tflops_sustained"],
                "source": "measured"}
    return {"hbm": 6650.0, "tensor_burst": 1590.0, "tensor": 1400.0, "source": "fallback"}


def dump_outputs(path, arrays):
    """Write each tensor of ``arrays`` (name -> tensor) as ``path/<name>.npy`` in float32.  A tensor of more than
    DUMP_SAMPLE entries is flattened and only the entries at DUMP_SAMPLE indices drawn with a fixed seed (kept in index
    order) are written: the same entries on every run, so dumps of two builds line up."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().to(torch.float32).cpu()
        if a.numel() > DUMP_SAMPLE:
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
            a = a.reshape(-1)[idx]
        np.save(os.path.join(path, name + ".npy"), a.numpy())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0=0.0):
        """Summary of the samples taken at or after wall-clock time t0 (the start of the measured load)."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for t, r in self.rows:
            if t < t0:
                continue
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the same training step on the host cores
# --------------------------------------------------------------------------------------------------------------------

def cpu_reference_arm(workload, steps, warmup, batch=None, components_too=False):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import torch
    import cpc_oracle_model as M
    w = WORKLOADS[workload]
    if w["cpu_batch"] is None:
        return None
    batch = batch or w["cpu_batch"]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    if workload == "raw_wave":
        model = M.OracleRawWave(w["visible"], w["prediction"])
        kw = dict(all_steps=False, kind="softplus", regularization=1.0)
    else:
        model = M.OracleE24(w["visible"], w["prediction"])
        kw = dict(all_steps=True, kind="linear", regularization=0.0)
    g = torch.Generator().manual_seed(1234)
    x = 0.1 * torch.randn(batch, model.item_length, generator=g)
    M.train_steps(model, [x] * warmup, **kw)
    t0 = time.perf_counter()
    M.train_steps(model, [x] * steps, **kw)
    dt = (time.perf_counter() - t0) / steps
    audio_s = batch * model.item_length / SR
    components = cpu_components(workload, batch, model.item_length) if components_too else None
    return {"value": audio_s / dt, "unit": "audio-s/s", "cores": cores, "kind": "port", "components": components,
            "sample": "%d steps of the same %s training step at batch %d (%.1f audio-s per step), torch CPU fp32, "
                      "%d threads, anomaly mode off" % (steps, workload, batch, audio_s, cores),
            "ms_per_step": dt * 1e3, "item_length": int(model.item_length)}


def cpu_components(workload, batch, item_length):
    """BASELINE.md section 4, item 4: the two stand-alone stages on the host cores -- PreprocessingModule.forward (CQT +
    log-power + phase) at the CPU batch, and the InfoNCE score + loss block forward + backward at the GPU's native size
    (B = 64), the largest the CPU path materialises comfortably ((B K)^2 scores)."""
    import torch
    import cpc_oracle as O
    w = WORKLOADS[workload]
    out = {}
    if workload != "raw_wave":
        plan = O.CqtPlan(16000, 30, 256, 32, 0.5, 128)
        x = 0.1 * torch.randn(batch, 1, item_length, generator=torch.Generator().manual_seed(1))
        O.preprocess(x, plan, phase=True)
        t0 = time.perf_counter()
        O.preprocess(x, plan, phase=True)
        dt = time.perf_counter() - t0
        out["cqt_scalogram_ms"] = dt * 1e3
        out["cqt_audio_s_per_s"] = batch * item_length / SR / dt
    k, e, b = w["prediction"], 512, 64
    all_steps, kind, reg = (False, "softplus", 1.0) if workload == "raw_wave" else (True, "linear", 0.0)
    g = torch.Generator().manual_seed(2)
    pred = (torch.randn(b, k, e, generator=g) / e ** 0.5).requires_grad_(True)
    tgt = torch.randn(b, e, k, generator=g).requires_grad_(True)
    for i in range(2):
        t0 = time.perf_counter()
        loss, _ = O.infonce_loss(pred, tgt, all_steps, kind, reg)
        loss.backward()
        dt = time.perf_counter() - t0
        pred.grad = tgt.grad = None
    out["infonce_fwd_bwd_ms"] = dt * 1e3
    out["infonce_shape"] = "B=%d K=%d E=%d %s %s" % (b, k, e, "all-steps" if all_steps else "per-step", kind)
    return out


def workload_config(workload, n_gpus, batch, item_length):
    w = WORKLOADS[workload]
    return {"workload": w["text"], "batch_per_gpu": batch, "global_batch": batch * n_gpus,
            "samples_per_item": item_length, "sample_rate": w.get("sr", SR), "parallelism": "dp%d" % n_gpus,
            "negatives": "per-GPU",
            "submission": ("whole step captured in CUDA graphs (cpc_b200.GraphedTrainStep)" if w.get("graph", True)
                           else "kernels submitted eagerly"),
            "l2": "activations (>300 MB per layer at batch 64) exceed the 126 MB L2; no explicit flush",
            "first_layer_dgrad": "skipped: the reference marks the scalogram requires_grad (contrastive_estimation_training"
                                 ".py:102) but only the gradient penalty reads that gradient; the CPU arm computes it",
            "library_math": "cuDNN / cuBLAS TF32 disabled (stock-PyTorch parts run fp32)",
            "filterbank_parity": "librosa.filters.constant_q restated, not pinned by the reference (DESIGN.md section 2)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = WORKLOADS[args.workload]
    if w["cpu_batch"] is None:
        emit({"impl": "reference", "unavailable": "no CPU port of workload %s (attention AR model)" % args.workload})
        return
    steps, warm = max(1, args.steps), max(1, args.warmup)
    r = cpu_reference_arm(args.workload, steps, warm)
    cfg = workload_config(args.workload, args.gpus, w["cpu_batch"], r["item_length"])
    cfg.update(submission="CPU port of the reference training step (oracle/), batch %d per step" % w["cpu_batch"],
               first_layer_dgrad="computed (as the reference does)", library_math="torch CPU fp32 (oneDNN)")
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "audio-s/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# --------------------------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------------------------

def build_workload(name, dev):
    """-> (model, preprocessing, trainer kwargs, learning rate) for a training-step workload."""
    import torch
    import cpc_b200
    from cpc_b200 import configs, ops
    w = WORKLOADS[name]
    if name == "raw_wave":
        enc = cpc_b200.AudioEncoder(dict(cpc_b200.encoder_default_dict))
        model = cpc_b200.AudioPredictiveCodingModel(enc, cpc_b200.AudioGRUModel(512, 256), enc_size=512, ar_size=256,
                                                    visible_steps=w["visible"], prediction_steps=w["prediction"]).to(dev)
        kw = dict(regularization=1.0, score_over_all_timesteps=False, score_function=cpc_b200.softplus_score_function,
                  preprocessing=None, prediction_steps=w["prediction"])
        return model, None, kw, 1e-4
    if name == "e29":
        with open(os.path.join(ROOT, "tests", "golden", "configs.json")) as fh:      # the reference's dicts as imported
            exp = configs.experiment_from_plain(json.load(fh)["e29"])
    else:
        exp = configs.experiment("e20" if name == "e20_bf16" else "e24")
    tc = dict(exp["training_config"], visible_steps=w["visible"], prediction_steps=w["prediction"])
    if name == "e20_bf16":
        ops.set_default_precision("bf16")
        exp["ar_model_config"]["sequence_length"] = max(exp["ar_model_config"]["sequence_length"], w["visible"])
    model, pre, _ = configs.setup_model(exp["cqt_config"], exp["encoder_config"], exp["ar_model_config"], tc, device=dev)
    kw = dict(regularization=tc["regularization"], score_over_all_timesteps=tc["score_over_all_timesteps"],
              score_function=tc["score_function"], preprocessing=pre, prediction_steps=tc["prediction_steps"],
              wasserstein_gradient_penalty=tc["wasserstein_gradient_penalty"],
              gradient_penalty_factor=tc["gradient_penalty_factor"])
    return model, pre, kw, tc["learning_rate"]


def ncu_traffic(key):
    """DRAM bytes per launch of the kernel behind ``key`` from the committed ncu capture -- only when that capture was made
    with exactly the kernel sources of this build (profiles/ncu_traffic.json carries the source digest)."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(path):
        return None, "no ncu capture committed"
    with open(path) as fh:
        t = json.load(fh)
    import build as _build
    if t.get("source_digest") != _build._digest():
        return None, "stale: profiles/ncu_traffic.json was captured from other kernel sources"
    entry = t.get("kernels", {}).get(key)
    if entry is None:
        return None, "kernel not in the committed ncu capture"
    return entry["dram_bytes_per_launch"], "ncu --set full, %s" % t.get("captured", "")


def run_ours(args):
    # stdout carries exactly one JSON line: NCCL's own banner (NCCL_DEBUG=VERSION) goes to stderr
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    import torch
    import torch.distributed as dist
    import cpc_b200
    from cpc_b200 import _lib, ddp, ops

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback (use --impl reference for the CPU arm)")
    rank, world, local = ddp.init_from_env("nccl")
    if world != args.gpus:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d; launch with torchrun for N>1" % (args.gpus, world))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    _lib.check(_lib.load().cpc_runtime_check(), "cpc_runtime_check")
    ops.strict_fp32_libraries()

    w = WORKLOADS[args.workload]
    torch.manual_seed(0)
    model, pre, tkw, lr = build_workload(args.workload, dev)
    ddp.broadcast_parameters(model, 0)
    length = int(model.item_length)
    b = int(args.batch or w["batch"])
    trainer = cpc_b200.ContrastiveEstimationTrainer(model=model, dataset=None, device=dev, verbose=False, **tkw)
    optimizer = trainer.make_optimizer(lr)                      # torch.optim.Adam -> cpc_b200.optim.Adam (one kernel per step)
    use_graph = not args.no_graph and w.get("graph", True)
    model.train()

    g = torch.Generator().manual_seed(1234 + rank)
    host_batches = [(0.1 * torch.randn(b, length, generator=g)).pin_memory() for _ in range(2)]
    dev_batches = [h.to(dev) for h in host_batches]

    def eager_step(batch):
        loss, max_score = trainer.loss_on_batch(batch)
        model.zero_grad(set_to_none=True)
        loss.backward()
        if world > 1:
            ddp.allreduce_gradients([p for p in model.parameters() if p.requires_grad], world)
        optimizer.step()
        return loss, max_score

    graphed, launches_per_step = None, None
    if use_graph:
        # the whole step (forward, backward, Adam) is captured once and replayed; count our launches per step while
        # capturing (a replay issues no host-side launch calls)
        _lib.reset_launch_count()
        graphed = cpc_b200.GraphedTrainStep(trainer, optimizer, (b, length), warmup=3)
        launches_per_step = _lib.launch_count() // 4            # 3 eager warm-up steps + the captured one

    def step(batch):
        return graphed(batch) if graphed is not None else eager_step(batch)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(k):
            fn(i)
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) / k

    # Every timed step trains from the seeded initial state: the weights and buffers as they are now (before the warm-up
    # steps) and a fresh optimizer state (zero moments and step count), restored on the device before the step and
    # outside its events.  The kernels reduce with float atomics, whose order differs from run to run, and a chain of
    # training steps amplifies such last-bit differences; from one fixed state a step does the same work as any other
    # and computes the same result in every run, up to the rounding of that one step.
    initial = [(t, t.detach().clone()) for m in (model, pre) if m is not None
               for t in list(m.parameters()) + list(m.buffers())]

    clocks = ClockSampler(local)
    clocks.start()                                              # nvidia-smi needs a moment to deliver its first sample
    for i in range(args.warmup):
        step(dev_batches[i % 2])
    torch.cuda.synchronize()
    opt_state = [v for st in optimizer.state.values() for v in st.values() if torch.is_tensor(v)]
    opt_state += [g["_step_state"] for g in optimizer.param_groups if torch.is_tensor(g.get("_step_state"))]
    state = [t for t, _ in initial] + opt_state
    saved = [v for _, v in initial] + [torch.zeros_like(v) for v in opt_state]

    def restore():
        with torch.no_grad():
            for t, v in zip(state, saved):
                t.copy_(v)
    _lib.reset_launch_count()
    t_load = time.time()
    barrier()
    events = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for i, (e0, e1) in enumerate(events):
        restore()
        e0.record()
        last_out = step(dev_batches[i % 2])
        e1.record()
    barrier()
    ms_dev = max_over_ranks(sum(e0.elapsed_time(e1) for e0, e1 in events)) / args.steps
    launches = launches_per_step * args.steps if graphed is not None else _lib.launch_count()
    dumped = None
    if args.dump_outputs and rank == 0:
        # device copies now: the steps below overwrite the graph's static outputs and the gradients.  The graphed
        # multi-rank step leaves the sum over ranks in .grad and lets cpc_b200.optim.Adam scale it by 1 / world; every
        # other path leaves the average there, which is what is written.
        params = [p for p in model.parameters() if p.requires_grad]
        scale = 1.0 / world if graphed is not None and world > 1 and isinstance(optimizer, cpc_b200.optim.Adam) else 1.0
        dumped = {"loss": last_out[0].clone(), "max_score": last_out[1].clone(),
                  "gradients": scale * torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).detach()
                                                  .reshape(-1) for p in params])}
    # K steps of ~14 ms are shorter than a few 100 ms sampling periods: keep the identical load running (untimed) until
    # ~0.6 s of it have been sampled.  The count derives from ms_dev (max over ranks), so every rank runs the same steps.
    clock_window = "timed region"
    n_extra = int(600.0 / max(ms_dev, 1e-3)) - args.steps
    if n_extra > 0:
        for i in range(n_extra):
            step(dev_batches[i % 2])
        torch.cuda.synchronize()
        clock_window = "timed region + %d identical untimed steps right after it" % n_extra
    clk = clocks.stop(t_load)
    clk["window"] = clock_window

    # end to end through the public API: pinned host batch -> device, full step, loss + max score read back
    last = {}

    # Every step's batch travels pinned host -> device inside the timed region.  Like a DataLoader with
    # pin_memory + non_blocking copies, the copy of batch i+1 is issued on a side stream while step i computes.
    copy_stream = torch.cuda.Stream(device=dev)
    staged = [torch.empty(b, length, device=dev) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]

    def prefetch(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[i % 2])             # the step that last read this staging buffer is done
            staged[i % 2].copy_(host_batches[i % 2], non_blocking=True)
            ready[i % 2].record(copy_stream)

    # The result of every step (loss, max score) is copied to pinned host memory and read by the host inside the timed
    # region -- one step late, like a training loop that logs asynchronously: the host reads step i-1 after it has
    # submitted step i, so the GPU is not idle while Python turns around (the last step is read before the clock stops).
    host_result = [torch.empty(2, dtype=torch.float32).pin_memory() for _ in range(2)]
    result_ready = [torch.cuda.Event() for _ in range(2)]

    def read_result(i):
        result_ready[i % 2].synchronize()
        last["v"] = host_result[i % 2].tolist()

    def e2e_step(i, n_steps=args.steps):
        if i == 0:
            prefetch(0)
        torch.cuda.current_stream(dev).wait_event(ready[i % 2])
        prefetch(i + 1)
        loss, mx = step(staged[i % 2])
        consumed[i % 2].record(torch.cuda.current_stream(dev))
        host_result[i % 2].copy_(torch.stack([loss.detach(), mx.detach()]), non_blocking=True)   # device -> host
        result_ready[i % 2].record(torch.cuda.current_stream(dev))
        if i > 0:
            read_result(i - 1)
        if i == n_steps - 1:
            read_result(i)
    for ev in consumed:
        ev.record(torch.cuda.current_stream(dev))
    e2e_step(0, 1)
    torch.cuda.synchronize()
    for ev in consumed:
        ev.record(torch.cuda.current_stream(dev))
    ms_e2e = timed(e2e_step, args.steps)

    # per-kernel times: CUDA events around each C-ABI call inside real (eager) steps on the launching stream
    prof = ops.KernelProfiler()
    with prof:
        for i in range(max(2, min(args.steps, 4))):
            eager_step(dev_batches[i % 2])
    torch.cuda.synchronize()
    top = prof.summary()

    sr = w.get("sr", SR)
    audio_s_step = world * b * length / sr
    value = audio_s_step / (ms_dev * 1e-3)
    e2e_value = audio_s_step / (ms_e2e * 1e-3)
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    if rank != 0:
        # no destroy_process_group / interpreter teardown: CUDA graphs holding captured NCCL work make both hang
        sys.stderr.flush()
        os._exit(0)
    peaks = measured_peaks()

    # kernel families (one CUDA kernel function serves several layer shapes)
    fams = {}
    for k in top:
        name = k["key"].split("[")[-1].rstrip("]") if "[" in k["key"] else k["key"].split(" ")[0]
        f = fams.setdefault(name, {"family": name, "ms": 0.0, "flops": 0.0, "bytes": 0.0, "launches": 0})
        f["ms"] += k["total_ms"]
        f["flops"] += k["flops_per_launch"] * k["count"]
        f["bytes"] += k["bytes_per_launch"] * k["count"]
        f["launches"] += k["count"]
    total_ms = sum(f["ms"] for f in fams.values()) or 1.0
    fam_list = sorted(fams.values(), key=lambda f: -f["ms"])
    for f in fam_list:
        f["share"] = f["ms"] / total_ms
        f["tflops"] = f["flops"] / (f["ms"] * 1e-3) / 1e12 if f["ms"] > 0 else 0.0
        f["gbs"] = f["bytes"] / (f["ms"] * 1e-3) / 1e9 if f["ms"] > 0 else 0.0

    # roofline: the single most expensive kernel = one entry point at ONE shape (total time over the profiled steps)
    roofline = None
    if top:
        dom = top[0]
        traffic, traffic_note = ncu_traffic(dom["key"])
        common = {"traffic": traffic, "traffic_source": traffic_note, "kernel": dom["key"], "avg_launch_ms": dom["avg_ms"],
                  "launches": dom["count"], "share_of_kernel_time": dom["share"]}
        if dom["flops_per_launch"] > 0:
            roofline = dict(common, bound="tensor", achieved=dom["tflops"], peak=peaks["tensor"], unit="TFLOP/s",
                            frac=dom["tflops"] / peaks["tensor"],
                            algorithmic_flops_per_launch=dom["flops_per_launch"],
                            peak_source=peaks["source"] + " bf16 dense cuBLAS, sustained",
                            mma_passes=1 if w["dtype"] == "bf16" else 3,
                            frac_of_mode_ceiling=dom["tflops"] * (1 if w["dtype"] == "bf16" else 3) / peaks["tensor"],
                            note="achieved = algorithmic FLOPs of the launch (conv: 2*Cout*Cin*kh*kw*B*OH*OW, taps that fall "
                                 "into zero padding included) / its average CUDA-event time; the fp32-faithful mode issues 3 "
                                 "bf16 MMAs per product, so the ceiling of `frac` is 1/3 there; frac_of_mode_ceiling = "
                                 "mma_passes * frac")
        else:
            roofline = dict(common, bound="hbm", achieved=dom["gbs"], peak=peaks["hbm"], unit="GB/s",
                            frac=dom["gbs"] / peaks["hbm"], algorithmic_bytes_per_launch=dom["bytes_per_launch"],
                            peak_source=peaks["source"] + " copy bandwidth",
                            note="achieved = algorithmic bytes (passes over the activation) / average CUDA-event time")

    # the metric's other two thirds: CQT HBM GB/s (+ dense-equivalent TFLOP/s), InfoNCE and conv TFLOP/s
    def agg(prefix):
        rows = [k for k in top if k["key"].startswith(prefix)]
        ms = sum(k["total_ms"] for k in rows)
        if ms <= 0:
            return None, None, None
        return (sum(k["flops_per_launch"] * k["count"] for k in rows) / (ms * 1e-3) / 1e12,
                sum(k["bytes_per_launch"] * k["count"] for k in rows) / (ms * 1e-3) / 1e9,
                ms / max(1, sum(k["count"] for k in rows)))
    cqt_tf, cqt_gbs, cqt_ms = agg("cpc_cqt_fwd")
    nce_f = agg("cpc_infonce_fwd")
    nce_b = agg("cpc_infonce_bwd")
    metrics = {
        "cqt_hbm_gbs": cqt_gbs, "cqt_hbm_frac": (cqt_gbs / peaks["hbm"]) if cqt_gbs else None,
        "cqt_dense_tflops": cqt_tf, "cqt_ms": cqt_ms,
        "cqt_note": "GB/s = (audio read once + scalogram written once) / time of the whole front-end call; the direct-form "
                    "filterbank is a dense contraction (2 100 FLOP/B), so it is bound by the tensor pipe, not by HBM",
        "infonce_fwd_tflops": nce_f[0], "infonce_bwd_tflops": nce_b[0],
        "infonce_fwd_ms": nce_f[2], "infonce_bwd_ms": nce_b[2],
        "infonce_note": "native size (%d candidates): latency-bound; the large-N numbers are --workload infonce_sweep" % (
            b * tkw["prediction_steps"] if tkw["score_over_all_timesteps"] else b),
        "conv_tflops_by_family": {f["family"]: f["tflops"] for f in fam_list if f["flops"] > 0 and "conv" in f["family"]},
        "conv_tensor_frac_by_family": {f["family"]: f["tflops"] / peaks["tensor"] for f in fam_list
                                       if f["flops"] > 0 and "conv" in f["family"]},
    }
    cpu = cpu_reference_arm(args.workload, 2, 1, components_too=True) if world == 1 else None
    line = {"metric": METRIC, "value": value, "unit": "audio-s/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": w["dtype"], "data": "synthetic",
            "config": workload_config(args.workload, world, b, length),
            "clocks": clk, "gpu_launches": launches,
            "e2e": {"value": e2e_value, "unit": "audio-s/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": b * length * 4, "d2h_bytes_per_step": 8, "last_loss": last["v"][0],
                    "result_read": "every step's (loss, max score) copied to pinned host memory and read by the host "
                                   "inside the timed region, one step late (asynchronous logging)"},
            "roofline": roofline, "metrics": metrics,
            "cpu_baseline": ({k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample", "components")} if cpu else None),
            "kernel_families": [{k: f[k] for k in ("family", "share", "ms", "launches", "tflops", "gbs")} for f in fam_list],
            "kernels": top[:40]}
    if world > 1:
        line["overlap"] = getattr(graphed, "overlap_description", None)
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped)
    emit(line)
    if world > 1:
        sys.stderr.flush()
        os._exit(0)


def run_infonce_sweep(args):
    """BASELINE configs[3]: fused InfoNCE forward + backward alone.  candidates N in 128...8192, K in 4...32, E = 512; per-step
    mode B = N, all-steps mode B = N / K; linear and softplus; regulariser 0 and 0.01; each point timed over --steps calls.
    Prints one JSON line whose `value` is the best fwd+bwd TFLOP/s of the sweep (algorithmic FLOPs = 4 x forward) and
    whose `sweep` lists every point."""
    import torch
    from cpc_b200 import _lib, ops
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback")
    dev = torch.device("cuda", 0)
    _lib.check(_lib.load().cpc_runtime_check(), "cpc_runtime_check")
    peaks = measured_peaks()
    e = 512
    points = []
    gen = torch.Generator(device=dev).manual_seed(0)
    for all_steps in (False, True):
        for k in (4, 16, 32):
            for n in (128, 512, 2048, 8192):
                bsz = n // k if all_steps else n
                if bsz < 2:
                    continue
                for kind, reg in (("linear", 0.0), ("softplus", 0.0), ("linear", 0.01)):
                    if reg and (n not in (2048, 8192) or k != 16):
                        continue
                    pred = (torch.randn(bsz, k, e, device=dev, generator=gen) / e ** 0.5).requires_grad_(True)
                    tgt = torch.randn(bsz, e, k, device=dev, generator=gen).requires_grad_(True)

                    def once():
                        loss = ops.infonce(pred, tgt, all_steps, kind, reg)[0]
                        loss.backward()
                        pred.grad = tgt.grad = None
                    for _ in range(2):
                        once()
                    torch.cuda.synchronize()
                    reps = args.steps
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(reps):
                        once()
                    e1.record()
                    torch.cuda.synchronize()
                    ms = e0.elapsed_time(e1) / reps
                    fwd = 2.0 * (bsz * k) ** 2 * e if all_steps else 2.0 * k * bsz * bsz * e
                    points.append({"mode": "all-steps" if all_steps else "per-step", "candidates": n, "K": k, "B": bsz,
                                   "score": kind, "reg": reg, "ms": ms, "tflops": 4.0 * fwd / (ms * 1e-3) / 1e12})
    best = max(points, key=lambda p: p["tflops"])
    emit({"metric": "InfoNCE fused score+loss fwd+bwd TFLOP/s (sweep best)", "value": best["tflops"], "unit": "TFLOP/s",
          "n_gpus": 1, "steps": args.steps, "warmup": 2, "ms_per_step": best["ms"], "higher_is_better": True, "scaling": "weak",
          "vs_baseline": None, "dtype": "f32", "data": "synthetic",
          "config": {"workload": "infonce_sweep: fused InfoNCE fwd+bwd, E=512, candidates 128-8192 x K 4-32 (BASELINE configs[3])",
                     "best_point": best},
          "roofline": {"bound": "tensor", "achieved": best["tflops"], "peak": peaks["tensor"], "unit": "TFLOP/s",
                       "frac": best["tflops"] / peaks["tensor"], "traffic": None,
                       "note": "algorithmic FLOPs = 4 x forward (recompute + dP + dZ); fp32-faithful mode: ceiling 1/3"},
          "sweep": points})


_RESULT_FD = None


def _claim_stdout():
    """stdout must carry exactly ONE JSON line, but libraries loaded later write banners to file descriptor 1 (NCCL
    prints "NCCL version ..." there at communicator creation).  Keep a private duplicate of the real stdout for the
    result line and point descriptor 1 (and sys.stdout) at stderr for everything else."""
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = sys.stderr


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="e24", choices=sorted(WORKLOADS) + ["infonce_sweep"])
    ap.add_argument("--batch", type=int, default=None, help="items per GPU (default: the workload's)")
    ap.add_argument("--no-graph", action="store_true", help="submit kernels eagerly instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed training step computed to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload == "infonce_sweep"):
        ap.error("--dump-outputs applies to the training-step workloads of --impl ours")
    args.warmup = max(3, args.warmup) if args.impl == "ours" else args.warmup
    if args.workload == "infonce_sweep":
        if args.impl == "reference":
            emit({"impl": "reference", "unavailable": "the reference cannot materialise the sweep's score tensors"})
        else:
            run_infonce_sweep(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

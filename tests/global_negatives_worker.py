"""Worker of tests/test_global_negatives.py: one process per rank, global negatives across data-parallel ranks.

  gloo (CPU, float64): ``ddp.gather_predictions`` and ``ddp.combine_shard_losses`` around a float64 stand-in for the
      rectangular InfoNCE loss.  The returned loss / max and the averaged parameter gradients must equal the global
      loss, max and gradients evaluated on the whole batch in one process.
  nccl (one rank per GPU, launched with torch.distributed.run):
      1. raw-wave model with global negatives, on the eager path of train() (loss_on_batch, backward,
         GradientBucketReducer) and on GraphedTrainStep: every rank's loss and max against the oracle's global ones (the
         oracle runs each shard's encoder separately and concatenates P and Z), the averaged gradients against the
         oracle's gradients of the global loss.
      2. e24 at the full item length: every rank's loss against the oracle's global loss.
"""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "constrastive-predictive-coding-audio_b200"), os.path.join(ROOT, "oracle")):
    sys.path.insert(0, p)
from cpc_b200 import ddp                                     # noqa: E402


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def rect_loss(p_all, z, offset, lam):
    """All-steps linear InfoNCE on the column block of rank `offset // b`: rows (d, k) of every item, columns (t, k') of
    this rank's items, positive of column (t, k') at row (offset + t, k')."""
    n, k, _ = p_all.shape
    b = z.shape[0]
    s = torch.einsum("dke,tel->dktl", p_all, z)                      # (n, K, b, K)
    flat = s.reshape(n * k, b * k)
    cols = torch.arange(b * k)
    loss = (torch.logsumexp(flat, 0) - flat[offset * k + cols, cols]).mean()
    return loss + lam * (s.mean(1) ** 2).mean(), s.max()


def main_gloo(init_file):
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dist.init_process_group("gloo", init_method="file://" + init_file, rank=rank, world_size=world)
    b, k, e, f, lam = 3, 4, 5, 6, 0.3
    gen = torch.Generator().manual_seed(5)
    x = torch.randn(world * b, f, generator=gen, dtype=torch.float64)
    wp0 = torch.randn(f, k * e, generator=gen, dtype=torch.float64) / f
    wz0 = torch.randn(f, e * k, generator=gen, dtype=torch.float64) / f

    def forward(xs, wp, wz):
        return torch.tanh(xs @ wp).view(-1, k, e), (xs @ wz).view(-1, e, k)

    # the global loss on one process
    wp, wz = wp0.clone().requires_grad_(True), wz0.clone().requires_grad_(True)
    p, z = forward(x, wp, wz)
    want, want_max = rect_loss(p, z, 0, lam)
    want.backward()
    # rank r: its shard, the gathered predictions, L_r, then the gradient average of data-parallel training
    mp, mz = wp0.clone().requires_grad_(True), wz0.clone().requires_grad_(True)
    p_r, z_r = forward(x[rank * b:(rank + 1) * b], mp, mz)
    loss_r, max_r = rect_loss(ddp.gather_predictions(p_r), z_r, rank * b, lam)
    loss, mx = ddp.combine_shard_losses(loss_r, max_r)
    assert abs(float(loss) - float(want)) < 1e-12 and float(mx) == float(want_max), (float(loss), float(want))
    loss.backward()
    for got, ref in ((mp.grad, wp.grad), (mz.grad, wz.grad)):
        dist.all_reduce(got)
        got /= world
        assert rel(got, ref) < 1e-12, rel(got, ref)
    # the mean of the shard losses is the global loss; a single shard's is not
    assert abs(float(loss_r) - float(want)) > 1e-6
    dist.barrier()
    print("RANK_OK %d" % rank, flush=True)


def main_nccl():
    import cpc_b200
    import cpc_oracle as O
    import cpc_oracle_model as OM
    rank, world, local = ddp.init_from_env("nccl")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    assert world >= 2

    # ---- 1. raw-wave model: eager train() path and GraphedTrainStep against the oracle's global loss ----------------
    chans = [16, 24, 24, 24, 32]
    torch.manual_seed(0)
    enc = cpc_b200.AudioEncoder({'strides': [5, 4, 2, 2, 2], 'kernel_sizes': [10, 8, 4, 4, 4], 'channel_count': chans,
                                 'bias': True})
    model = cpc_b200.AudioPredictiveCodingModel(enc, cpc_b200.AudioGRUModel(32, 16), enc_size=32, ar_size=16,
                                                visible_steps=9, prediction_steps=4).to(dev)
    ddp.broadcast_parameters(model, 0)
    per = 6
    g = torch.Generator().manual_seed(78)
    global_batch = 0.1 * torch.randn(per * world, model.item_length, generator=g)
    shard = ddp.shard_batch(global_batch, rank, world)
    trainer = cpc_b200.ContrastiveEstimationTrainer(model=model, dataset=None, device=dev, regularization=1.0,
                                                    score_over_all_timesteps=False,
                                                    score_function=cpc_b200.softplus_score_function, prediction_steps=4,
                                                    verbose=False, global_negatives=True)
    oracle = OM.OracleRawWave(9, 4, channels=chans, ar_size=16)
    own = dict(model.named_parameters())
    name_map = {}
    for i in range(5):
        name_map["encoder.layers.%d.weight" % i], name_map["encoder.layers.%d.bias" % i] = "convs.%d.weight" % i, "convs.%d.bias" % i
    for leaf in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"):
        name_map["autoregressive_model.gruCell." + leaf] = "gru." + leaf
    name_map["prediction_model.weight"] = "predict.weight"
    theirs = dict(oracle.named_parameters())
    assert set(name_map) == set(own) and set(name_map.values()) == set(theirs)
    with torch.no_grad():
        for k, v in name_map.items():
            theirs[v].copy_(own[k].detach().cpu())
    outs = [oracle(global_batch[r * per:(r + 1) * per]) for r in range(world)]
    pred = torch.cat([o[0] for o in outs])
    tgt = torch.cat([o[1] for o in outs])
    want_loss, want_max = O.infonce_loss(pred, tgt, False, "softplus", 1.0)
    want_loss.backward()

    def check(tag, loss, mx, grads):
        assert abs(loss - float(want_loss)) < 1e-3 * abs(float(want_loss)), (tag, loss, float(want_loss))
        assert abs(mx - float(want_max)) < 1e-3 * max(1.0, abs(float(want_max))), (tag, mx, float(want_max))
        for k, v in name_map.items():
            assert rel(grads[k], theirs[v].grad) < 3e-3, (tag, k, rel(grads[k], theirs[v].grad))

    # eager, as train() runs a step (on a side stream, without keeping the loss: see nccl_parity_worker.py)
    reducer = ddp.GradientBucketReducer(model)
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        loss_t, mx_t = trainer.loss_on_batch(shard.to(dev))
        model.zero_grad(set_to_none=True)
        loss_t.backward()
        reducer.finish()
        eager = (loss_t.item(), mx_t.item(), {k: v.grad.detach().clone() for k, v in own.items()})
        del loss_t, mx_t
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize(dev)
    reducer.remove()
    check("eager", *eager)
    # graphed step with SGD(lr=0): weights stay, the flat buffer holds the averaged gradients
    model.zero_grad(set_to_none=True)
    opt = torch.optim.SGD(model.parameters(), lr=0.0)
    step = cpc_b200.GraphedTrainStep(trainer, opt, (per, model.item_length), warmup=2)
    assert "captured inside" in step.overlap_description, step.overlap_description
    loss, mx = step(shard.to(dev))
    torch.cuda.synchronize()
    check("graphed", loss.item(), mx.item(), {k: v.grad for k, v in own.items()})
    step.remove_hooks()

    # ---- 2. e24 at the full item length: every rank returns the oracle's global loss -----------------------------------
    exp = cpc_b200.configs.experiment("e24")
    tc = exp["training_config"]
    torch.manual_seed(0)
    model, pre, _ = cpc_b200.configs.setup_model(exp["cqt_config"], exp["encoder_config"], exp["ar_model_config"], tc,
                                                 device=dev)
    OM.reseed_parameters(model.named_parameters())
    per = 2
    audio = OM.e24_audio(per * world, model.item_length, seed=4322)
    shard = ddp.shard_batch(audio, rank, world)
    trainer = cpc_b200.ContrastiveEstimationTrainer(model=model, dataset=None, device=dev,
                                                    regularization=tc["regularization"],
                                                    score_over_all_timesteps=tc["score_over_all_timesteps"],
                                                    score_function=tc["score_function"], preprocessing=pre,
                                                    prediction_steps=tc["prediction_steps"], verbose=False,
                                                    global_negatives=True)
    model.train()
    oracle = OM.OracleE24(60, 16)
    OM.reseed_parameters(oracle.named_parameters(), OM.oracle_e24_name_map())
    oracle.train()
    with torch.no_grad():
        outs = [oracle(audio[r * per:(r + 1) * per]) for r in range(world)]    # BatchNorm statistics per shard
        want_e24, _ = O.infonce_loss(torch.cat([o[0] for o in outs]), torch.cat([o[1] for o in outs]), True, "linear",
                                     tc["regularization"])
        loss_e24, _ = trainer.loss_on_batch(shard.to(dev))
    value = loss_e24.item()
    assert abs(value - float(want_e24)) < 1e-3 * abs(float(want_e24)), (value, float(want_e24))
    dist.barrier()
    print("RANK_OK %d (raw-wave global loss %.6f, e24 global loss %.6f vs oracle %.6f, %s)"
          % (rank, float(want_loss), value, float(want_e24), step.overlap_description), flush=True)


if __name__ == "__main__":
    try:
        if sys.argv[1] == "gloo":
            main_gloo(sys.argv[2])
        else:
            main_nccl()
    except BaseException:                                         # noqa: BLE001 -- report compactly, never hang the launcher
        import traceback
        print("RANK_FAILED %s\n%s" % (os.environ.get("RANK"), traceback.format_exc()[-2500:]), flush=True)
        os._exit(1)
    os._exit(0)                                                   # skip interpreter teardown of graphs holding NCCL work

"""Worker of tests/test_sharded_validate.py: one process per GPU (torch.distributed.run, NCCL).

e24 with BatchNorm running statistics that differ between the ranks.  ``validate(shard_over_ranks=True)`` must return on
every rank the values rank 0 computes by validating the whole batches alone with its own statistics, identical on all
ranks, and leave every rank's own buffers as they were.
"""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "constrastive-predictive-coding-audio_b200"), os.path.join(ROOT, "oracle")):
    sys.path.insert(0, p)
from cpc_b200 import ddp                                     # noqa: E402


class Items(torch.utils.data.Dataset):
    def __init__(self, items):
        self.items = items

    def __len__(self):
        return self.items.shape[0]

    def __getitem__(self, i):
        return self.items[i]

    def get_example_count_per_file(self):
        return [len(self)]


def main():
    import cpc_b200
    import cpc_oracle_model as OM
    rank, world, local = ddp.init_from_env("nccl")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    assert world >= 2
    exp = cpc_b200.configs.experiment("e24")
    tc = exp["training_config"]
    torch.manual_seed(0)
    model, pre, _ = cpc_b200.configs.setup_model(exp["cqt_config"], exp["encoder_config"], exp["ar_model_config"], tc,
                                                 device=dev)
    OM.reseed_parameters(model.named_parameters())
    ddp.broadcast_parameters(model, 0)
    # diverged running statistics: every rank moves its buffers by its own amount
    gen = torch.Generator().manual_seed(100 + rank)
    with torch.no_grad():
        for name, b in model.named_buffers():
            if name.endswith("running_mean"):
                b.add_(0.2 * torch.randn(b.shape, generator=gen).to(dev))
            elif name.endswith("running_var"):
                b.mul_(torch.empty(b.shape).uniform_(0.5, 2.0, generator=gen).to(dev))
    own = {n: b.detach().clone() for n, b in model.named_buffers()}
    assert any(n.endswith("running_mean") for n in own)
    per_batch = 8
    val = Items(OM.e24_audio(2 * per_batch, model.item_length, seed=977))          # two validation batches
    trainer = cpc_b200.ContrastiveEstimationTrainer(model=model, dataset=None, validation_set=val, device=dev,
                                                    score_over_all_timesteps=tc["score_over_all_timesteps"],
                                                    score_function=tc["score_function"], preprocessing=pre,
                                                    prediction_steps=tc["prediction_steps"], verbose=False)
    sharded = trainer.validate(batch_size=per_batch, num_workers=0, shard_over_ranks=True)
    for n, b in model.named_buffers():
        assert torch.equal(b, own[n]), n                                         # own statistics restored
    assert model.training
    alone = trainer.validate(batch_size=per_batch, num_workers=0)                 # this rank, the whole batches
    flat = torch.cat([sharded[0], sharded[1], torch.tensor([sharded[2]], device=dev, dtype=torch.float32), sharded[3]])
    everyone = flat.new_empty((world, flat.numel()))
    dist.all_gather_into_tensor(everyone, flat.contiguous())
    assert all(torch.equal(everyone[0], everyone[r]) for r in range(world)), everyone   # bit-identical on every rank
    ref = torch.cat([alone[0], alone[1], torch.tensor([alone[2]], device=dev, dtype=torch.float32), alone[3]])
    rank0 = ref.clone()
    dist.broadcast(rank0, src=0)                                                  # rank 0's single-process values
    k = tc["prediction_steps"]
    n = per_batch * k if tc["score_over_all_timesteps"] else per_batch
    losses, acc, score = flat[:k], flat[k:2 * k], float(flat[2 * k])
    assert float((losses - rank0[:k]).abs().max()) < 1e-4 * max(1.0, float(rank0[:k].abs().max())), (losses, rank0[:k])
    # Accuracy: at most one hit per slot apart over the two batches (1 / (2n)).  The shard path forwards 4 items, the
    # reference 8, and the convolution families choose their tiles and splits by batch size, so the predictions agree
    # only to rounding; a row whose two best scores are that close can change its arg-max.  The emulated-shard tests
    # in test_sharded_validate.py, which feed both paths the same predictions, require exact hit counts.
    assert float((acc - rank0[k:2 * k]).abs().max()) <= 1.0 / (2 * n) + 1e-7, (acc, rank0[k:2 * k])
    assert abs(score - float(rank0[2 * k])) < 1e-4 * max(1.0, abs(float(rank0[2 * k]))), (score, float(rank0[2 * k]))
    if rank > 0:                                                                  # the statistics matter
        assert float((ref[:k] - rank0[:k]).abs().max()) > 1e-4, "diverged BatchNorm statistics changed nothing"
    dist.barrier()
    print("RANK_OK %d (losses %s, accuracy %s, mean score %.6f)" % (rank, losses.tolist(), acc.tolist(), score),
          flush=True)


if __name__ == "__main__":
    try:
        main()
    except BaseException:                                         # noqa: BLE001 -- report compactly, never hang the launcher
        import traceback
        print("RANK_FAILED %s\n%s" % (os.environ.get("RANK"), traceback.format_exc()[-2500:]), flush=True)
        os._exit(1)
    os._exit(0)

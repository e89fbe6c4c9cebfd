"""Worker of tests/test_device_loader.py: one process per GPU (torch.distributed.run, NCCL).

Rank 0 writes a WAV folder; every rank then iterates ``DeviceBatchLoader(rank, world)`` over a seeded sampler and checks
that each batch it gets is its contiguous shard of the single-process batch ``torch.stack([ds[i] for i in batch])``.
Then ``validate(shard_over_ranks=True, device_loading=True)`` must equal rank 0's unsharded ``validate()``.
"""
import os
import random
import sys
import tempfile

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "constrastive-predictive-coding-audio_b200"), os.path.join(ROOT, "oracle"),
          os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
from cpc_b200 import ddp                                     # noqa: E402


def main():
    import cpc_b200
    from cpc_b200.audio_dataset import AudioDataset
    from cpc_b200.device_loader import DeviceBatchLoader
    from cpc_b200.sampler import FileBatchSampler
    from test_device_loader import make_folder
    import pathlib

    rank, world, local = ddp.init_from_env("nccl")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    assert world >= 2
    torch.manual_seed(0)
    enc = cpc_b200.AudioEncoder({'strides': [5, 4, 2, 2, 2], 'kernel_sizes': [10, 8, 4, 4, 4],
                                 'channel_count': [16, 24, 24, 24, 32], 'bias': True})
    model = cpc_b200.AudioPredictiveCodingModel(enc, cpc_b200.AudioGRUModel(32, 16), enc_size=32, ar_size=16,
                                                visible_steps=9, prediction_steps=4).to(dev)
    ddp.broadcast_parameters(model, 0)
    n = model.item_length
    with tempfile.TemporaryDirectory() as tmp:
        path = [os.path.join(tmp, "r0")] if rank == 0 else [None]
        dist.broadcast_object_list(path, src=0)               # one folder, written by rank 0 (same host)
        root = pathlib.Path(path[0])
        if rank == 0:
            make_folder(root, [3 * n + 17, n // 2, n // 3 + 5, 4 * n, 2 * n + 1, n + 3], 2, 3, seed=70)
        dist.barrier()
        ds = AudioDataset(root, item_length=n, unique_length=n // 2)
        per, batch_size = 4, 4 * world
        random.seed(5)                                        # rank 0's `random` draws the batches
        sampler = FileBatchSampler(ds.get_example_count_per_file(), batch_size=batch_size, drop_last=True)
        recorded = []

        class Recording(torch.utils.data.Sampler):
            def __iter__(self):
                for b in sampler:
                    recorded.append(list(b))
                    yield b

            def __len__(self):
                return len(sampler)
        loader = DeviceBatchLoader(ds, Recording(), dev, rank=rank, world=world)
        got = []
        for _ in range(2):
            got.extend(b.cpu() for b in loader)
        everyone = [None] * world
        dist.all_gather_object(everyone, recorded)
        batches = everyone[0]                                  # only rank 0 iterates the sampler
        assert len(got) == len(batches) >= 4, (len(got), len(batches))
        for b, want_idx in zip(got, batches):
            want = torch.stack([ds[i] for i in want_idx[rank * per:(rank + 1) * per]])
            assert torch.equal(b, want), want_idx
        trainer = cpc_b200.ContrastiveEstimationTrainer(model=model, dataset=ds, validation_set=ds, device=dev,
                                                        score_function=cpc_b200.softplus_score_function,
                                                        prediction_steps=4, verbose=False)
        sharded = trainer.validate(batch_size=batch_size, shard_over_ranks=True, device_loading=True)
        alone = trainer.validate(batch_size=batch_size, num_workers=0)
        flat = torch.cat([sharded[0], sharded[1], torch.tensor([sharded[2]], device=dev), sharded[3]])
        ref = torch.cat([alone[0], alone[1], torch.tensor([alone[2]], device=dev), alone[3]])
        dist.broadcast(ref, src=0)                             # rank 0's single-process values
        k = 4
        assert float((flat[:k] - ref[:k]).abs().max()) < 1e-4 * max(1.0, float(ref[:k].abs().max())), (flat, ref)
        # the shard path forwards batch/W items, so predictions agree to rounding only (see sharded_validate_worker.py)
        assert float((flat[k:2 * k] - ref[k:2 * k]).abs().max()) <= 1.0 / batch_size + 1e-7, (flat, ref)
        assert abs(float(flat[2 * k] - ref[2 * k])) < 1e-4 * max(1.0, abs(float(ref[2 * k])))
        dist.barrier()
    print("RANK_OK %d (%d batches)" % (rank, len(got)), flush=True)


if __name__ == "__main__":
    try:
        main()
    except BaseException:                                         # noqa: BLE001 -- report compactly, never hang the launcher
        import traceback
        print("RANK_FAILED %s\n%s" % (os.environ.get("RANK"), traceback.format_exc()[-2500:]), flush=True)
        os._exit(1)
    os._exit(0)

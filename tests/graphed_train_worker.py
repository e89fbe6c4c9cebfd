"""Worker of tests/test_graphed_train.py: one process per GPU (torch.distributed.run, NCCL).

1. ``train(cuda_graph=True)`` against eager ``train()`` over 3 steps of a WAV folder, with per-GPU and with global
   negatives: the logged losses agree on every rank.
2. A NaN loss on rank 1 only (per-GPU negatives): both ranks return at the same step, and neither rank's weights nor
   Adam state moved in the NaN step.
"""
import os
import pathlib
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
    from test_device_loader import make_folder
    from test_graphed_train import RecordingLogger, _adam_state

    rank, world, local = ddp.init_from_env("nccl")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    assert world >= 2

    def setup(root, global_negatives, logger):
        torch.manual_seed(0)
        enc = cpc_b200.AudioEncoder({'strides': [5, 4, 2, 2, 2], 'kernel_sizes': [10, 8, 4, 4, 4],
                                     'channel_count': [16, 24, 24, 24, 32], 'bias': True})
        model = cpc_b200.AudioPredictiveCodingModel(enc, cpc_b200.AudioGRUModel(32, 16), enc_size=32, ar_size=16,
                                                    visible_steps=9, prediction_steps=4).to(dev)
        ds = AudioDataset(root, item_length=model.item_length, unique_length=model.item_length // 2)
        trainer = cpc_b200.ContrastiveEstimationTrainer(model=model, dataset=ds, device=dev, logger=logger,
                                                        score_function=cpc_b200.softplus_score_function,
                                                        prediction_steps=4, verbose=False,
                                                        global_negatives=global_negatives)
        made = []
        plain = trainer.make_optimizer
        trainer.make_optimizer = lambda lr, **kw: made.append(plain(lr, **kw)) or made[-1]
        return trainer, made

    with tempfile.TemporaryDirectory() as tmp:
        path = [os.path.join(tmp, "r0")] if rank == 0 else [None]
        dist.broadcast_object_list(path, src=0)               # one folder, written by rank 0 (same host)
        root = pathlib.Path(path[0])
        n = cpc_b200.AudioPredictiveCodingModel(                  # the item length of setup's model
            cpc_b200.AudioEncoder({'strides': [5, 4, 2, 2, 2], 'kernel_sizes': [10, 8, 4, 4, 4],
                                   'channel_count': [16, 24, 24, 24, 32], 'bias': True}),
            cpc_b200.AudioGRUModel(32, 16), enc_size=32, ar_size=16, visible_steps=9, prediction_steps=4).item_length
        if rank == 0:
            make_folder(root, [3 * n + 17, n // 2, n // 3 + 5, 4 * n, 2 * n + 1, n + 3, 5 * n, 2 * n], 1, 2, seed=80)
        dist.barrier()
        batch_size = 4 * world

        # 1. graphed against eager losses, per-GPU and global negatives
        for global_negatives in (False, True):
            losses = []
            for cuda_graph in (False, True):
                logger = RecordingLogger()
                trainer, _ = setup(root, global_negatives, logger)
                random.seed(5)                                 # rank 0's `random` draws the batches
                trainer.train(batch_size=batch_size, epochs=3, lr=1e-3, max_steps=3, device_loading=True,
                              cuda_graph=cuda_graph)
                assert trainer.training_step == 3 and logger.steps == [0, 1, 2], logger.steps
                losses.append(logger.loss_meter.values)
            eager, graphed = losses
            for a, b in zip(eager, graphed):
                assert abs(a - b) <= 1e-4 * max(1.0, abs(a)), (global_negatives, eager, graphed)

        # 2. NaN on rank 1 only
        stop_at = 2
        poison = torch.ones((), device=dev)
        snap = {}
        holder = {}

        def on_log(step):
            if step == stop_at - 1:
                snap["state"] = _adam_state(holder["made"][0])
                if rank == 1:
                    poison.fill_(float("nan"))
        trainer, made = setup(root, False, RecordingLogger(on_log))
        holder["made"] = made
        trainer.model.register_forward_hook(lambda mod, inp, out: (out[0] * poison,) + tuple(out[1:]))
        random.seed(5)
        trainer.train(batch_size=batch_size, epochs=3, lr=1e-3, device_loading=True, cuda_graph=True)
        assert trainer.training_step == stop_at, trainer.training_step
        assert trainer.last_loss != trainer.last_loss
        after = _adam_state(made[0])
        assert len(after) == len(snap["state"])
        for i, (x, y) in enumerate(zip(snap["state"], after)):
            assert torch.equal(x, y), i
        steps = [None] * world
        dist.all_gather_object(steps, trainer.training_step)
        assert steps == [stop_at] * world, steps
        dist.barrier()
    print("RANK_OK %d" % rank, flush=True)


if __name__ == "__main__":
    try:
        main()
    except BaseException:                                         # noqa: BLE001 -- report compactly, never hang the launcher
        import traceback
        print("RANK_FAILED %s\n%s" % (os.environ.get("RANK"), traceback.format_exc()[-2500:]), flush=True)
        os._exit(1)
    os._exit(0)

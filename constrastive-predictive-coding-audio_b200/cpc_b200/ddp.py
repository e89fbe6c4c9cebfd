"""Data-parallel plumbing: one process per GPU, gradients averaged with bucketed NCCL all-reduces that are
issued from autograd hooks while backward is still running (SURVEY.md 8e).

The reference uses single-process ``nn.DataParallel`` (setup_functions.py:112-115).  Here every rank owns a
contiguous slice of each batch -- the same dim-0 chunking ``DataParallel.scatter`` applies.

Negatives.  By default they stay on the rank (north star): each rank scores its shard against its own predictions and
the forward pass needs no collective at all; the loss is the mean of W shard losses, not the reference's.  Opt-in,
``ContrastiveEstimationTrainer(global_negatives=True)`` reproduces what DataParallel computes on the outputs it gathers
onto one GPU: every target is ranked against the predictions of the whole global batch.  Each rank all-gathers the
predictions (``gather_predictions``), scores its own targets against them (a rectangular ``ops.infonce`` call) and
back-propagates its shard loss L_r; the backward of the gather reduce-scatters the prediction gradients with SUM.
Since mean_r L_r is the global loss, that sum is W times the global gradient of this rank's predictions, and the
usual averaging of the parameter gradients over W leaves exactly the global gradient.  BatchNorm statistics stay per
rank, as in DataParallel's replicas.
"""
import os

import torch
import torch.distributed as dist


def init_from_env(backend=None):
    """Initialise torch.distributed from RANK / WORLD_SIZE / LOCAL_RANK / MASTER_* (torchrun).  Returns
    (rank, world, local_rank); single-process when WORLD_SIZE is unset or 1."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29500")
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(local)
            dist.init_process_group(backend=backend, rank=rank, world_size=world,
                                    device_id=torch.device("cuda", local))
        else:
            dist.init_process_group(backend=backend, rank=rank, world_size=world)
    return rank, world, local


def shard_batch(batch, rank, world):
    """Rank r's slice of a global batch: ``batch[r*B/W:(r+1)*B/W]`` (DataParallel.scatter chunking)."""
    if world == 1:
        return batch
    b = batch.shape[0]
    if b % world:
        raise ValueError("global batch %d is not divisible by world size %d" % (b, world))
    per = b // world
    return batch[rank * per:(rank + 1) * per]


class ShardedBatchSampler(torch.utils.data.Sampler):
    """Wraps a batch sampler for one-process-per-GPU training: rank 0 iterates the wrapped sampler (so its use of
    Python's ``random`` is exactly the single-process one), the epoch's index lists are broadcast, and every rank
    yields only its contiguous shard ``batch[r*B/W:(r+1)*B/W]`` of each batch -- ranks agree on the global batch and
    load 1/W of it."""

    def __init__(self, batch_sampler, rank, world, group=None):
        self.batch_sampler, self.rank, self.world, self.group = batch_sampler, rank, world, group

    def __iter__(self):
        payload = [list(map(list, iter(self.batch_sampler)))] if self.rank == 0 else [None]
        if self.world > 1:
            dist.broadcast_object_list(payload, src=0, group=self.group)
        for batch in payload[0]:
            if len(batch) % self.world:
                raise ValueError("global batch %d is not divisible by world size %d" % (len(batch), self.world))
            per = len(batch) // self.world
            yield batch[self.rank * per:(self.rank + 1) * per]

    def __len__(self):
        return len(self.batch_sampler)


class _GatherPredictions(torch.autograd.Function):
    """Forward: all-gather of the ranks' (b, ...) tensors into (W*b, ...) in rank order.  Backward: reduce-scatter (SUM)
    of the gathered gradient, each rank keeping its own rows.  Both are plain synchronous collectives, ordered with the
    current stream, so they can be captured in a CUDA graph (GraphedTrainStep)."""

    @staticmethod
    def forward(ctx, x, group):
        ctx.group = group
        world = dist.get_world_size(group)
        x = x.contiguous()
        out = x.new_empty((world * x.shape[0],) + tuple(x.shape[1:]))
        dist.all_gather_into_tensor(out, x, group=group)
        return out

    @staticmethod
    def backward(ctx, grad):
        world = dist.get_world_size(ctx.group)
        grad = grad.contiguous()
        out = grad.new_empty((grad.shape[0] // world,) + tuple(grad.shape[1:]))
        # NCCL calls on one communicator must be issued in the same order on every rank.  This one is issued when
        # autograd reaches the gather node, right after the InfoNCE node's backward: the gather is the newest node on
        # every path from the predictions to the loss, so no parameter gradient is final yet and no gradient-bucket
        # all-reduce hook has fired.  Keep the gather directly in front of the InfoNCE call to keep it so.
        dist.reduce_scatter_tensor(out, grad, op=dist.ReduceOp.SUM, group=ctx.group)
        return out, None


def gather_predictions(x, group=None):
    """All ranks' ``x`` concatenated along dim 0 in rank order, differentiable: the gradient that reaches each rank's
    ``x`` is the SUM over ranks of the gradients of the gathered tensor at its rows."""
    return _GatherPredictions.apply(x, group)


def combine_shard_losses(loss_r, max_r, group=None):
    """(L_r, max_r) of each rank -> (loss, max) with the value of mean_r L_r and of max_r max_r on every rank, from one
    all-gather of a 2-vector.  The loss keeps the gradient of L_r: ``L_r + (mean - L_r).detach()``."""
    world = dist.get_world_size(group)
    local = torch.stack([loss_r.detach().reshape(()), max_r.detach().reshape(())]).to(loss_r.dtype)
    both = local.new_empty(2 * world)
    dist.all_gather_into_tensor(both, local, group=group)
    both = both.view(world, 2)
    return loss_r + (both[:, 0].mean() - loss_r).detach(), both[:, 1].max()


def broadcast_parameters(module, src=0):
    if not dist.is_initialized() or dist.get_world_size() == 1:
        return
    for t in list(module.parameters()) + list(module.buffers()):
        dist.broadcast(t.data, src=src)


def allreduce_gradients(params, world, bucket_mb=64.0, group=None):
    """Synchronous variant used after a CUDA-graph replay (the graph holds forward + backward only): average the
    .grad buffers across ranks in flat buckets, in place."""
    if world == 1 or not dist.is_initialized():
        return
    limit = int(bucket_mb * 1024 * 1024)
    bucket, size = [], 0

    def flush():
        if not bucket:
            return
        flat = torch.cat([g.reshape(-1) for g in bucket])
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
        flat.div_(world)
        offset = 0
        for g in bucket:
            n = g.numel()
            g.copy_(flat[offset:offset + n].view_as(g))
            offset += n

    for p in params:
        if p.grad is None:
            continue
        bucket.append(p.grad)
        size += p.grad.numel() * p.grad.element_size()
        if size >= limit:
            flush()
            bucket, size = [], 0
    flush()


class GradientBucketReducer:
    """Averages ``.grad`` across ranks.  Parameters are packed into buckets of ~``bucket_mb`` in reverse
    registration order (the order autograd produces them); when the last gradient of a bucket has been
    accumulated the bucket is flattened and its all-reduce launched asynchronously, overlapping the rest of
    backward.  ``finish()`` waits, divides by the world size and scatters the result back into ``.grad``."""

    def __init__(self, module, bucket_mb=25.0, process_group=None):
        self.group = process_group
        self.world = dist.get_world_size(process_group) if dist.is_initialized() else 1
        self.params = [p for p in module.parameters() if p.requires_grad]
        limit = int(bucket_mb * 1024 * 1024)
        self.buckets, current, size = [], [], 0
        for p in reversed(self.params):
            current.append(p)
            size += p.numel() * p.element_size()
            if size >= limit:
                self.buckets.append(current)
                current, size = [], 0
        if current:
            self.buckets.append(current)
        self._bucket_of = {}
        for bi, bucket in enumerate(self.buckets):
            for p in bucket:
                self._bucket_of[p] = bi
        self._pending = [0] * len(self.buckets)
        self._inflight = []
        self._hooks = []
        self.launched_during_backward = 0
        if self.world > 1:
            for p in self.params:
                self._hooks.append(p.register_post_accumulate_grad_hook(self._on_grad))
        self.reset()

    def reset(self):
        self._pending = [len(b) for b in self.buckets]
        self._inflight = []
        self.launched_during_backward = 0

    def _on_grad(self, param):
        bi = self._bucket_of[param]
        self._pending[bi] -= 1
        if self._pending[bi] == 0:
            self._launch(bi)
            self.launched_during_backward += 1

    def _launch(self, bi):
        grads = [p.grad for p in self.buckets[bi] if p.grad is not None]
        if not grads:
            return
        flat = torch.cat([g.reshape(-1) for g in grads])
        work = dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group, async_op=True)
        self._inflight.append((work, flat, grads))

    def finish(self):
        """Call after ``loss.backward()`` and before ``optimizer.step()``."""
        if self.world == 1:
            return
        for bi, left in enumerate(self._pending):
            if left > 0:                      # parameters that received no gradient this step
                self._launch(bi)
        for work, flat, grads in self._inflight:
            work.wait()
            flat.div_(self.world)
            offset = 0
            for g in grads:
                n = g.numel()
                g.copy_(flat[offset:offset + n].view_as(g))
                offset += n
        self.reset()

    def remove(self):
        for h in self._hooks:
            h.remove()
        self._hooks = []

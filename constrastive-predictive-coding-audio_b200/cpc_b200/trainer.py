"""``ContrastiveEstimationTrainer`` with the fused InfoNCE kernels behind the reference's API.

Constructor, ``train`` and ``validate`` signatures follow contrastive_estimation_training.py:36-269.  The
three named score functions stay importable; when the trainer is given ``linear_score_function``,
``softplus_score_function`` or ``difference_score_function`` the whole block ``score -> logsumexp -> loss ->
regulariser -> max`` (:106-122, :141, :166) is ONE fused forward kernel family and one backward, and the (B,K,B,K)
score tensor never exists (nor, for the difference kind, the (B,K,E,B,K) tensor of differences).  Any other score
function runs the literal block.

Multi-GPU: one process per GPU.  Each rank trains on its contiguous slice of every batch, negatives stay on
the rank, gradients are averaged by ``ddp.GradientBucketReducer`` while backward runs.
"""
import math
import time

import torch
import torch.nn.functional as F
import torch.optim
import torch.utils.data

from . import ddp, ops, optim
from .sampler import FileBatchSampler


def softplus_score_function(predicted_z, targets):
    """(B,K,E),(B,E,K) -> (B,K,B,K) materialised scores; kept for API compatibility (dreaming etc.).  The
    trainer recognises this function object and uses the fused kernel instead of calling it."""
    return F.softplus(torch.tensordot(predicted_z, targets, dims=([2], [1])))


def linear_score_function(predicted_z, targets):
    return torch.tensordot(predicted_z, targets, dims=([2], [1]))


def difference_score_function(predicted_z, targets):
    diff = predicted_z.unsqueeze(3).unsqueeze(4) - targets.permute(1, 0, 2).unsqueeze(0).unsqueeze(1)
    return 1 / torch.sum(diff ** 2, dim=2)


_FUSED_KINDS = {linear_score_function: "linear", softplus_score_function: "softplus",
                difference_score_function: "difference"}


def reference_loss_from_scores(scores, batch_size, prediction_steps, all_steps, regularization):
    """The literal loss block for score functions the fused kernel does not know (:108-122,141)."""
    if all_steps:
        noise = torch.logsumexp(scores.reshape(-1, batch_size, prediction_steps), dim=0)
        valid = torch.diagonal(torch.diagonal(scores, dim1=0, dim2=2), dim1=0, dim2=1)
    else:
        scores = torch.diagonal(scores, dim1=1, dim2=3).permute(0, 2, 1).contiguous()
        noise = torch.logsumexp(scores.view(-1, batch_size, prediction_steps), dim=0)
        valid = torch.diagonal(scores, dim1=0, dim2=2).permute(1, 0)
    loss = torch.mean(-torch.mean(valid - noise, dim=1))
    loss = loss + regularization * torch.mean(torch.mean(scores, dim=1) ** 2)
    return loss, scores.max()


class ContrastiveEstimationTrainer:
    def __init__(self, model, dataset, logger=None, device=None, regularization=1., validation_set=None,
                 test_task_set=None, prediction_noise=0.01, optimizer=torch.optim.Adam, file_batch_size=1,
                 score_over_all_timesteps=False, score_function=softplus_score_function,
                 wasserstein_gradient_penalty=False, gradient_penalty_factor=10., preprocessing=None, ar_size=256,
                 prediction_steps=16, verbose=True):
        self.model = model
        self.ar_size = ar_size
        self.prediction_steps = prediction_steps
        self.dataset = dataset
        self.logger = logger
        self.device = device
        self.regularization = regularization
        self.validation_set = validation_set
        self.test_task_set = test_task_set
        self.training_step = 0
        self.print_out_scores = False
        self.prediction_noise = prediction_noise
        self.optimizer = optimizer
        self.file_batch_size = file_batch_size
        self.score_over_all_timesteps = score_over_all_timesteps
        self.score_function = score_function
        self.wasserstein_gradient_penalty = wasserstein_gradient_penalty
        self.gradient_penalty_factor = gradient_penalty_factor
        self.preprocessing = preprocessing
        self.verbose = verbose
        self.rank, self.world = 0, 1
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            self.rank, self.world = torch.distributed.get_rank(), torch.distributed.get_world_size()
        self.last_loss = None
        self.last_max_score = None
        if ops.get_default_precision() == "fp32":
            ops.strict_fp32_libraries()                         # no TF32 in the cuDNN / cuBLAS parts (AR model, W_k)
        if verbose:
            print("use score function", self.score_function)

    # -- one step -----------------------------------------------------------------------------------
    def loss_on_batch(self, batch):
        """batch: (B, L) audio on the device -> (loss, max_score).  Rows are this rank's items."""
        batch = batch.unsqueeze(1)
        if self.preprocessing is not None:
            batch = self.preprocessing(batch)
            # The reference marks the scalogram as requiring grad (:102) but only the gradient penalty ever
            # reads that gradient; without the penalty the first layer's data gradient is dead work, so it is
            # not requested here (identical losses and parameter gradients).  The flag is only ever raised: with a
            # trainable filterbank the scalogram is a non-leaf that already requires grad, and assigning False to
            # it would raise.
            if self.wasserstein_gradient_penalty and not batch.requires_grad:
                batch.requires_grad_(True)
        kind = _FUSED_KINDS.get(self.score_function)
        if self.wasserstein_gradient_penalty:
            return self._loss_with_gradient_penalty(batch, kind)
        predicted_z, targets, _, _ = self.model(batch)
        if kind is not None:
            loss, max_score, _, _ = ops.infonce(predicted_z, targets, self.score_over_all_timesteps, kind,
                                                self.regularization)
        else:
            scores = self.score_function(predicted_z, targets)
            loss, max_score = reference_loss_from_scores(scores, predicted_z.shape[0], self.prediction_steps,
                                                         self.score_over_all_timesteps, self.regularization)
        return loss, max_score

    def _loss_with_gradient_penalty(self, batch, kind):
        """:144-158: loss + factor * mean((||d sum(scores) / d scalogram||_2 over channels - 1)^2).  The penalty is
        differentiated a second time by loss.backward(), so the encoder runs in second-order mode: convolutions on the
        B200 kernels with differentiable dgrad / wgrad nodes, BN / ReLU / pooling as the literal modules.  The InfoNCE
        term still goes through the fused kernels; only the penalty's sum(scores) uses the materialised scores."""
        with ops.second_order():
            predicted_z, targets, _, _ = self.model(batch)
            scores = self.score_function(predicted_z, targets)
            if not self.score_over_all_timesteps:
                scores = torch.diagonal(scores, dim1=1, dim2=3).permute(0, 2, 1).contiguous()
            if kind is not None:
                loss, max_score, _, _ = ops.infonce(predicted_z, targets, self.score_over_all_timesteps, kind,
                                                    self.regularization)
            else:
                loss, max_score = reference_loss_from_scores(self.score_function(predicted_z, targets),
                                                             predicted_z.shape[0], self.prediction_steps,
                                                             self.score_over_all_timesteps, self.regularization)
            batch_grad = torch.autograd.grad(outputs=torch.sum(scores), inputs=batch, create_graph=True,
                                             retain_graph=True, only_inputs=True)
            penalty = ((batch_grad[0].norm(2, dim=1) - 1) ** 2).mean() * self.gradient_penalty_factor
        return loss + penalty, max_score

    def make_optimizer(self, lr, **kwargs):
        """``self.optimizer(self.model.parameters(), lr=lr)`` (:84); the stock ``torch.optim.Adam`` class is replaced
        by the single-kernel ``cpc_b200.optim.Adam`` (same arithmetic and state_dict) when the model is on a GPU."""
        cls = self.optimizer
        if cls is torch.optim.Adam and all(p.is_cuda for p in self.model.parameters()):
            cls = optim.Adam
        return cls(self.model.parameters(), lr=lr, **kwargs)

    def _any_rank_nan(self, loss):
        """True when the loss is NaN on ANY rank (one host sync; one tiny all-reduce when world > 1), so that all
        ranks leave train() together instead of one returning and the others blocking in the next all-reduce."""
        flag = torch.isnan(loss.detach()).to(torch.float32).reshape(1)
        if self.world > 1:
            torch.distributed.all_reduce(flag, op=torch.distributed.ReduceOp.MAX)
        return bool(flag.item())

    def train(self, batch_size=32, epochs=10, lr=0.0001, continue_training_at_step=0, num_workers=1, max_steps=None,
              profile=False):
        self.model.train()
        optimizer = self.make_optimizer(lr)
        sampler = FileBatchSampler(index_count_per_file=self.dataset.get_example_count_per_file(),
                                   batch_size=batch_size, file_batch_size=self.file_batch_size, drop_last=True)
        reducer = None
        if self.world > 1:
            # every rank starts from rank 0's weights and sees rank 0's batches: the sampler draws from rank 0's
            # (unseeded, global) `random` state exactly as the single-process reference does, the index lists are
            # broadcast, and each rank loads only its contiguous shard of every batch (DataParallel.scatter chunking)
            ddp.broadcast_parameters(self.model)
            sampler = ddp.ShardedBatchSampler(sampler, self.rank, self.world)
            reducer = ddp.GradientBucketReducer(self.model)
        dataloader = torch.utils.data.DataLoader(self.dataset, batch_sampler=sampler, num_workers=num_workers,
                                                 pin_memory=True)
        self.training_step = continue_training_at_step
        try:
            for current_epoch in range(epochs):
                if self.verbose:
                    print("epoch", current_epoch)
                with torch.autograd.profiler.profile(use_device='cuda', enabled=profile) as prof:
                    for batch in iter(dataloader):
                        batch = batch.to(device=self.device, non_blocking=True)
                        loss, max_score = self.loss_on_batch(batch)
                        # :124-133 -- the reference leaves BEFORE backward / optimizer.step, so weights and optimizer
                        # state stay finite
                        if self._any_rank_nan(loss):
                            print("nan loss")
                            print("returned with nan loss at step", self.training_step)
                            self.last_loss = float("nan")
                            return
                        self.model.zero_grad()
                        loss.backward()
                        if reducer is not None:
                            reducer.finish()
                        optimizer.step()
                        # one host read per step for (loss, max score)
                        loss_value, max_value = torch.stack([loss.detach(), max_score.detach()]).tolist()
                        self.last_loss, self.last_max_score = loss_value, max_value
                        if self.logger is not None:
                            self.logger.loss_meter.update(loss_value)
                            self.logger.score_meter.update(max_value)
                            self.logger.log(self.training_step)
                        elif self.verbose:
                            print("loss at step step " + str(self.training_step) + ":", loss_value)
                        self.training_step += 1
                        if max_steps is not None and self.training_step >= max_steps:
                            return prof
        finally:
            if reducer is not None:
                reducer.remove()

    # -- validation: fused metrics kernel for the known score functions, literal block otherwise --------
    def validate(self, batch_size=64, num_workers=1, max_steps=None):
        if self.validation_set is None:
            print("No validation set")
            return 0, 0
        self.model.eval()
        sampler = FileBatchSampler(index_count_per_file=self.validation_set.get_example_count_per_file(),
                                   batch_size=batch_size, file_batch_size=8, drop_last=True, seed=0)
        loader = torch.utils.data.DataLoader(self.validation_set, batch_sampler=sampler, num_workers=num_workers,
                                             pin_memory=False)
        k = self.prediction_steps
        total_losses = torch.zeros(k, device=self.device)
        total_accurate = torch.zeros(k, device=self.device)
        n = batch_size * k if self.score_over_all_timesteps else batch_size
        template = torch.arange(0, n, dtype=torch.long, device=self.device)
        template = template.view(batch_size, k) if self.score_over_all_timesteps else template.unsqueeze(1).repeat(1, k)
        total_score = 0
        max_steps = len(loader) if max_steps is None else min(max_steps, len(loader))
        with torch.no_grad():
            for step, batch in enumerate(iter(loader)):
                batch = batch.to(device=self.device).unsqueeze(1)
                if self.preprocessing is not None:
                    batch = self.preprocessing(batch)
                predicted_z, targets, _, _ = self.model(batch)
                kind = _FUSED_KINDS.get(self.score_function)
                if kind is not None and predicted_z.is_cuda:
                    losses, accuracy, mean_score = ops.infonce_validate(predicted_z, targets,
                                                                        self.score_over_all_timesteps, kind)
                    total_losses += losses
                    total_accurate += accuracy
                    total_score += mean_score.item()
                    if step + 1 >= max_steps:
                        break
                    continue
                scores = self.score_function(predicted_z, targets)
                if self.score_over_all_timesteps:
                    noise = torch.logsumexp(scores.reshape(-1, batch_size, k), dim=0)
                    valid = torch.diagonal(torch.diagonal(scores, dim1=0, dim2=2), dim1=0, dim2=1)
                else:
                    scores = torch.diagonal(scores, dim1=1, dim2=3).permute(0, 2, 1).contiguous()
                    noise = torch.logsumexp(scores.view(-1, batch_size, k), dim=0)
                    valid = torch.diagonal(scores, dim1=0, dim2=2).permute(1, 0)
                losses = -torch.mean(valid - noise, dim=0)
                best = torch.argmax(scores.reshape(batch_size, k, -1), dim=2)
                accuracy = torch.sum(torch.eq(template, best), dim=0).type_as(batch) / n
                total_losses += losses
                total_accurate += accuracy
                total_score += torch.mean(scores).item()
                if step + 1 >= max_steps:
                    break
        del loader
        total_losses /= max_steps
        total_accurate /= max_steps
        total_score /= max_steps
        mutual_information_lb = math.log(n) - total_losses
        self.model.train()
        return total_losses, total_accurate, total_score, mutual_information_lb


class GraphedTrainStep:
    """One full training step (preprocessing -> model -> fused InfoNCE -> backward -> optimizer) captured once into a
    CUDA graph and replayed: the ~380 kernel launches of a step are submitted with one call, so the GPU never waits
    for Python between kernels.  Everything the step touches lives at fixed addresses (the static input batch, the
    parameters, their .grad buffers, the optimizer state and every workspace come from the graph's private pool).

        step = GraphedTrainStep(trainer, optimizer, (B, L))      # optimizer must be capturable (Adam(capturable=True))
        loss, max_score = step(batch)                            # batch: (B, L) device or pinned-host tensor

    With more than one rank the gradient all-reduce is PART of the graph and overlaps backward: every ``.grad`` is a
    view into one flat buffer laid out in reverse registration order (the order autograd finishes them), cut into a few
    contiguous buckets; when the last gradient of a bucket has been accumulated, a post-accumulate hook forks a
    communication stream and all-reduces that bucket in place (NCCL, captured), while the main stream goes on with the
    backward pass of the earlier layers.  The optimizer joins the communication stream and reads the summed gradients
    straight from the flat buffer (scaled by 1 / world): no flatten / un-flatten copies.  For e24 the AR model and the
    prediction head (70 % of the bytes) are reduced under the ~8 ms of encoder backward that follow them; only the
    last bucket (the first encoder blocks, < 1 MB) is exposed.  If the NCCL build cannot be captured the step falls back
    to two graphs around one eager all-reduce (``overlap_description`` says which)."""

    def __init__(self, trainer, optimizer, batch_shape, warmup=3, bucket_mb=12.0):
        self.trainer, self.optimizer = trainer, optimizer
        self.world = trainer.world
        dev = trainer.device
        self.static_batch = torch.zeros(batch_shape, dtype=torch.float32, device=dev)
        self.params = [p for p in trainer.model.parameters() if p.requires_grad]
        self.update_graph = None
        self.overlap_description = "single rank: no collective"
        self._hooks = []
        if self.world > 1:
            self._setup_flat_gradients(bucket_mb)
        # Warm-up steps outside the capture create the optimizer state, cuDNN plans, the NCCL communicator and the
        # allocator blocks the capture must not contain; they run on a scratch copy of the training state, which is
        # restored afterwards so that building the graph leaves model and optimizer exactly as they were.
        modules = [trainer.model] + ([trainer.preprocessing] if trainer.preprocessing is not None else [])
        tensors = [t for m in modules for t in list(m.parameters()) + list(m.buffers())]
        saved = [t.detach().clone() for t in tensors]
        saved_state = {p: {k: v.detach().clone() for k, v in optimizer.state.get(p, {}).items() if torch.is_tensor(v)}
                       for p in self.params}
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(max(1, warmup)):
                self._step_body()
        torch.cuda.current_stream(dev).wait_stream(side)
        with torch.no_grad():
            for t, s in zip(tensors, saved):
                t.copy_(s)
            for p in self.params:
                for k, v in optimizer.state.get(p, {}).items():
                    if torch.is_tensor(v):
                        old = saved_state[p].get(k)
                        v.copy_(old) if old is not None else v.zero_()
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        if self.world == 1:
            optimizer.zero_grad(set_to_none=True)
            with torch.cuda.graph(self.graph):
                self.loss, self.max_score = self._step_body()
            return
        # "thread_local": ProcessGroupNCCL's watchdog thread polls events of earlier (eager) collectives with
        # cudaEventQuery; under the default "global" capture mode such a call from ANY thread invalidates the capture
        torch.distributed.barrier()
        torch.cuda.synchronize(dev)
        try:
            with torch.cuda.graph(self.graph, capture_error_mode="thread_local"):
                self.loss, self.max_score = self._step_body()
            self.overlap_description = ("NCCL all-reduce of %d gradient buckets captured inside the step's CUDA graph on a "
                                        "communication stream forked from backward (bucket bytes: %s)"
                                        % (len(self.buckets), [4 * (hi - lo) for lo, hi, _ in self.buckets]))
        except Exception as exc:                                   # noqa: BLE001 -- e.g. an NCCL that cannot be captured
            torch.cuda.synchronize(dev)
            self._build_two_graphs(repr(exc))

    # -- multi-rank plumbing ---------------------------------------------------------------------------------------
    def _setup_flat_gradients(self, bucket_mb):
        dev = self.trainer.device
        order = list(reversed(self.params))
        offsets, total = [], 0
        for p in order:                                          # every segment starts on a 16-byte boundary
            offsets.append(total)
            total += (p.numel() + 3) // 4 * 4
        self.flat = torch.zeros(total, dtype=torch.float32, device=dev)
        for p, o in zip(order, offsets):
            p.grad = self.flat[o:o + p.numel()].view_as(p)
        limit = int(bucket_mb * 1024 * 1024 / 4)
        self.buckets, lo, members = [], 0, []
        for p, o in zip(order, offsets):
            members.append(p)
            hi = o + (p.numel() + 3) // 4 * 4
            if hi - lo >= limit:
                self.buckets.append((lo, hi, members))
                lo, members = hi, []
        if members:
            self.buckets.append((lo, total, members))
        self._bucket_of = {p: i for i, (_, _, ms) in enumerate(self.buckets) for p in ms}
        self._pending = [0] * len(self.buckets)
        self.comm_stream = torch.cuda.Stream(device=dev)
        self._serial = False                                     # True in the two-graph fallback: hooks do nothing
        for p in self.params:
            self._hooks.append(p.register_post_accumulate_grad_hook(self._on_gradient))

    def _on_gradient(self, param):
        if self._serial:
            return
        i = self._bucket_of[param]
        self._pending[i] -= 1
        if self._pending[i] == 0:
            self._reduce_bucket(i)

    def _reduce_bucket(self, i):
        lo, hi, _ = self.buckets[i]
        self.comm_stream.wait_stream(torch.cuda.current_stream(self.trainer.device))
        with torch.cuda.stream(self.comm_stream):
            torch.distributed.all_reduce(self.flat[lo:hi], op=torch.distributed.ReduceOp.SUM)

    def _step_body(self):
        """forward + backward (+ overlapped bucket all-reduces) + optimizer; identical eager (warm-up) and captured."""
        trainer, optimizer = self.trainer, self.optimizer
        if self.world == 1:
            optimizer.zero_grad(set_to_none=True)
            loss, max_score = trainer.loss_on_batch(self.static_batch)
            loss.backward()
            optimizer.step()
            return loss.detach(), max_score.detach()
        self.flat.zero_()                                        # gradients accumulate in place into the flat views
        self._pending = [len(ms) for _, _, ms in self.buckets]
        loss, max_score = trainer.loss_on_batch(self.static_batch)
        loss.backward()
        if self._serial:
            return loss.detach(), max_score.detach()
        for i, left in enumerate(self._pending):                 # parameters that received no gradient this step
            if left > 0:
                self._reduce_bucket(i)
        torch.cuda.current_stream(self.trainer.device).wait_stream(self.comm_stream)
        self._optimizer_step()
        return loss.detach(), max_score.detach()

    def _optimizer_step(self):
        if isinstance(self.optimizer, optim.Adam):               # reads the summed gradients in place, scaled by 1/W
            self.optimizer.step(grad_scale=1.0 / self.world)
        else:
            self.flat.div_(self.world)
            self.optimizer.step()

    def _build_two_graphs(self, why):
        """Fallback: forward + backward | eager all-reduce of the whole flat buffer | optimizer."""
        self._serial = True
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, capture_error_mode="thread_local"):
            self.loss, self.max_score = self._step_body()
        self.update_graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.update_graph, pool=self.graph.pool(), capture_error_mode="thread_local"):
            self._optimizer_step()
        self.overlap_description = "not overlapped: two graphs around one eager NCCL all-reduce (capture failed: %s)" % why

    def remove_hooks(self):
        for h in self._hooks:
            h.remove()
        self._hooks = []

    def __call__(self, batch):
        self.static_batch.copy_(batch, non_blocking=True)
        self.graph.replay()
        if self.update_graph is not None:
            torch.distributed.all_reduce(self.flat, op=torch.distributed.ReduceOp.SUM)
            self.update_graph.replay()
        return self.loss, self.max_score


class DeterministicSampler(torch.utils.data.Sampler):
    """contrastive_estimation_training.py:363-382: single indices of ``data_source`` in a pseudo-random order that is
    the same on every iteration (Python's ``random`` re-seeded with ``seed`` each time)."""

    def __init__(self, data_source, seed=0):
        self.data_source = data_source
        self.seed = seed

    def __iter__(self):
        import random
        order = list(range(len(self.data_source)))
        random.seed(self.seed)
        random.shuffle(order)
        return iter(order)

    def __len__(self):
        return len(self.data_source)

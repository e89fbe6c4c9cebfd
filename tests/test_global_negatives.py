"""Global negatives across data-parallel ranks: the rectangular (shard) InfoNCE problem of the C-ABI's _ex entry points,
its host wiring, the gather / reduce-scatter autograd Function (CPU, gloo), W shards emulated on one B200 against the
float64 oracle of the global batch, and the trainer option on one and on two GPUs."""
import ctypes
import math
import os
import subprocess
import sys

import pytest
import torch

import cpc_oracle as O
from conftest import rel_err

DEV = "cuda:0"
HERE = os.path.dirname(os.path.abspath(__file__))
WORKER = os.path.join(HERE, "global_negatives_worker.py")


def _align(n, a):
    return (n + a - 1) // a * a


def _params(lib_mod, b, k, e, all_steps, kind=0, reg=0.0):
    q = lib_mod.InfoNceParams()
    q.batch, q.steps, q.enc, q.all_steps, q.score_kind, q.regularization = b, k, e, int(all_steps), kind, reg
    q.tgt_stride_b, q.tgt_stride_e, q.tgt_stride_k = e * k, k, 1
    return q


def _shard(lib_mod, pred_batch, offset):
    sh = lib_mod.InfoNceShard()
    sh.pred_batch, sh.target_offset = pred_batch, offset
    return sh


# ---------------------------------------------------------------------------------------------------
# CPU: ABI, workspace sizes, host mirror, trainer constructor, gloo
# ---------------------------------------------------------------------------------------------------

def test_shard_entry_points_reject_bad_shards_before_the_device(built_lib):
    from cpc_b200 import _lib
    lib = _lib.load()
    q = _params(_lib, 4, 3, 8, True)
    fwd = lambda sh: lib.cpc_infonce_fwd_ex(None, None, None, None, ctypes.byref(q), sh, None, 0, None)   # noqa: E731
    bwd = lambda sh: lib.cpc_infonce_bwd_ex(None, None, None, None, None, None, ctypes.byref(q), sh, None, 0,  # noqa: E731
                                            None)
    for pred_batch, offset in ((3, 0), (6, 3), (6, -1), (4, 1), (1 << 29, 0)):
        sh = ctypes.byref(_shard(_lib, pred_batch, offset))
        assert fwd(sh) == -1 and bwd(sh) == -1, (pred_batch, offset)
        for which in (0, 1, 2):
            assert lib.cpc_infonce_workspace_bytes_ex(ctypes.byref(q), sh, which) == 0
    for pred_batch, offset in ((6, 2), (6, 0), (4, 0)):                         # valid: fail on the null pointers
        sh = ctypes.byref(_shard(_lib, pred_batch, offset))
        assert fwd(sh) == -7 and bwd(sh) == -7
        assert lib.cpc_infonce_workspace_bytes_ex(ctypes.byref(q), sh, 0) > 0
        assert lib.cpc_infonce_workspace_bytes_ex(ctypes.byref(q), sh, 2) == 0  # validation takes no shard
    assert fwd(None) == -7 and bwd(None) == -7
    for which in (0, 1, 2):                                                     # NULL and {batch, 0}: the square call
        plain = lib.cpc_infonce_workspace_bytes(ctypes.byref(q), which)
        assert lib.cpc_infonce_workspace_bytes_ex(ctypes.byref(q), None, which) == plain
    for which in (0, 1):
        assert lib.cpc_infonce_workspace_bytes_ex(ctypes.byref(q), ctypes.byref(_shard(_lib, 4, 0)), which) == \
            lib.cpc_infonce_workspace_bytes(ctypes.byref(q), which)
    assert lib.cpc_abi_version() == _lib.ABI_VERSION == 7


def test_shard_workspace_sizes_show_the_kernel_path(built_lib):
    """e24's shard shape (b = 64, K = 16, E = 512, all-steps) with 2 ranks: the tcgen05 path with its forward row
    split; the difference kind at the same shape and a small per-step shard: the CUDA-core kernels."""
    from cpc_b200 import _lib
    lib = _lib.load()
    b, k, e, w = 64, 16, 512, 2
    q = _params(_lib, b, k, e, True)
    sh = ctypes.byref(_shard(_lib, w * b, b))
    rows, cols = w * b * k, b * k                                               # 2048 prediction rows, 1024 columns
    planes = rows * e * 4 + cols * e * 4                                        # bf16 hi + lo of each operand
    rsplit = min(rows // 128, 148 // (cols // 128))                             # 16 CTAs per column tile
    ncta, nblk = (cols // 128) * rsplit, cols // 256
    umma_fwd = planes + _align((ncta + nblk) * 16, 256) + 2 * _align(rsplit * cols * 4, 256) + cols * 4 + 2048
    assert lib.cpc_infonce_workspace_bytes_ex(ctypes.byref(q), sh, 0) == umma_fwd
    assert lib.cpc_infonce_workspace_bytes_ex(ctypes.byref(q), sh, 1) == planes + 2048
    # difference kind: CUDA-core forward scratch (64-row tiles: 32 of them x 1024 columns of (max, sum-exp), the
    # positives' scores, 16 x 32 CTAs x (max, sum, reg), 4 combine blocks), no backward workspace
    q.score_kind = _lib.SCORE_DIFFERENCE
    core = 2 * 32 * cols * 4 + cols * 4 + 16 * 32 * 12 + 256
    assert lib.cpc_infonce_workspace_bytes_ex(ctypes.byref(q), sh, 0) == core
    assert lib.cpc_infonce_workspace_bytes_ex(ctypes.byref(q), sh, 1) == 0
    # per-step shard of 12 items among 48, lambda != 0: the (rows x columns) regulariser sums of the CUDA-core kernels
    q = _params(_lib, 12, 5, 40, False, _lib.SCORE_LINEAR, 0.01)
    assert lib.cpc_infonce_workspace_bytes_ex(ctypes.byref(q), ctypes.byref(_shard(_lib, 48, 24)), 1) == \
        _align(48 * 12 * 4, 256)


def test_ops_and_trainer_map_shard_calls():
    from cpc_b200 import ops, trainer
    pred, z = torch.zeros(8, 2, 5), torch.zeros(4, 5, 3)
    assert ops._nce_shard(pred[:4], z[:, :, -2:], 0) is None
    for all_steps, pairs_e in ((True, 8 * 2 * 4 * 2 * 5), (False, 2 * 8 * 4 * 5)):
        p = ops._nce_params(pred, z[:, :, -2:], all_steps, "linear", 0.0, "fp32")
        sh = ops._nce_shard(pred, z[:, :, -2:], 4)
        assert (p.batch, p.steps, p.enc, sh.pred_batch, sh.target_offset) == (4, 2, 5, 8, 4)
        assert ops._nce_flops(p, sh) == 2 * pairs_e and ops._nce_bwd_flops(p, sh) == 6 * pairs_e
        assert "x8" in ops._nce_key("cpc_infonce_fwd_ex", p, sh)
    common = dict(model=None, dataset=None, verbose=False, global_negatives=True)
    with pytest.raises(ValueError):
        trainer.ContrastiveEstimationTrainer(score_function=lambda p, t: trainer.linear_score_function(p, t), **common)
    with pytest.raises(ValueError):
        trainer.ContrastiveEstimationTrainer(score_function=trainer.linear_score_function,
                                             wasserstein_gradient_penalty=True, **common)
    t = trainer.ContrastiveEstimationTrainer(score_function=trainer.difference_score_function, **common)
    assert t.global_negatives and t.world == 1


def test_gather_reduce_scatter_function_gives_the_global_gradient_gloo(tmp_path):
    """Two CPU processes over gloo, float64: the averaged gradients of the shard losses equal the global loss's."""
    env = dict(os.environ, WORLD_SIZE="2")
    init = str(tmp_path / "init")
    procs = [subprocess.Popen([sys.executable, WORKER, "gloo", init], env=dict(env, RANK=str(r)),
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = []
    for pr in procs:
        try:
            outs.append(pr.communicate(timeout=240)[0])
        except subprocess.TimeoutExpired:
            for q in procs:
                q.kill()
            raise
    text = "\n".join(outs)
    assert all(pr.returncode == 0 for pr in procs), text[-3000:]
    assert "RANK_OK 0" in text and "RANK_OK 1" in text, text[-3000:]


# ---------------------------------------------------------------------------------------------------
# GPU: W shards emulated on one device
# ---------------------------------------------------------------------------------------------------

class _SquaredDistances(torch.autograd.Function):
    """D[r, c] = |p_r - z_c|^2 summed from explicit differences (cdist without the norm expansion).  Backward in closed
    form, dP = 2 (rowsum(G) P - G Z), dZ = 2 (colsum(G) Z - G^T P): cdist's own backward holds an (N, M, E) buffer."""

    @staticmethod
    def forward(ctx, p, z):
        ctx.save_for_backward(p, z)
        return torch.cdist(p, z, compute_mode="donot_use_mm_for_euclid_dist") ** 2

    @staticmethod
    def backward(ctx, g):
        p, z = ctx.saved_tensors
        return 2 * (g.sum(1, keepdim=True) * p - g @ z), 2 * (g.sum(0, keepdim=True).t() * z - g.t() @ p)


@pytest.fixture
def oracle(monkeypatch):
    """cpc_oracle with ``scores_full`` extended by kind='difference' (as in test_difference_score.py), without the
    (B,K,E,B,K) difference tensor, which would not fit at the larger batches here."""
    base = O.scores_full

    def scores_full(pred, targets, kind='linear'):
        if kind != 'difference':
            return base(pred, targets, kind)
        b, k, e = pred.shape
        d = _SquaredDistances.apply(pred.reshape(b * k, e), targets.permute(0, 2, 1).reshape(-1, e))
        return (1 / d).view(b, k, targets.shape[0], k)
    monkeypatch.setattr(O, "scores_full", scores_full)
    return O


@pytest.fixture(scope="module")
def cpc(built_lib):
    import cpc_b200
    assert cpc_b200._lib.load().cpc_runtime_check() == 0, "device is not a B200 (sm_100)"
    return cpc_b200


# (b, K, E) per shard: e24's shard (tcgen05 in all-steps mode), 128 items per step (tcgen05 in per-step mode without
# regulariser), and a small ragged shape (CUDA-core kernels)
SHAPES = {"tensor_all": (64, 16, 512, True), "tensor_step": (128, 4, 128, False), "core_all": (12, 5, 40, True),
          "core_step": (12, 5, 40, False)}


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("kind", ["linear", "softplus", "difference"])
def test_shards_reproduce_the_global_problem(cpc, oracle, kind, shape, world, precision):
    """For r in 0..W-1 the rectangular call on (P_all, Z_r, offset r*b): mean of the shard losses = global loss, max of
    the maxima = global max, sum of the d P_all = W x global d P, d Z_r = W x the global d Z_r; strided targets."""
    b, k, e, all_steps = SHAPES[shape]
    n = world * b
    gen = torch.Generator().manual_seed(1000 * world + b + k)
    pred = torch.randn(n, k, e, generator=gen) / math.sqrt(e)
    z = torch.randn(n, e, k + 3, generator=gen) / math.sqrt(e)                 # targets = strided view z[:, :, -k:]
    if kind == "difference":
        pred = pred + z[:, :, -k:].permute(0, 2, 1)                             # distances of order 1
    tol = 1e-3 if precision == "fp32" or kind == "difference" else 1e-2
    p64, t64 = pred.to(DEV, torch.float64), z[:, :, -k:].to(DEV, torch.float64)
    for reg in (0.0, 0.01):
        want_loss, want_max, want_dp, want_dz = oracle.infonce_with_grads(p64, t64, all_steps, kind, reg)
        want_loss0 = oracle.infonce_loss(p64, t64, all_steps, kind, 0.0)[0]
        s = oracle.scores_full(p64, t64, kind)
        s = s if all_steps else torch.diagonal(s, dim1=1, dim2=3)
        want_mean, score_scale = s.mean(), float(s.abs().mean())             # linear scores average to ~0
        del s
        pg = pred.to(DEV).requires_grad_(True)
        zs = z.to(DEV)
        losses, maxima, losses0, means, dz = [], [], [], [], []
        for r in range(world):
            zr = zs[r * b:(r + 1) * b].clone().requires_grad_(True)
            loss, mx, loss0, mean_s = cpc.ops.infonce(pg, zr[:, :, -k:], all_steps, kind, reg, precision=precision,
                                                      target_offset=r * b)
            (3.0 * loss).backward()                                              # non-unit upstream gradient
            losses.append(loss.item()); maxima.append(mx.item()); losses0.append(loss0.item()); means.append(mean_s.item())
            assert float(zr.grad[:, :, :-k].abs().max()) == 0.0
            dz.append(zr.grad[:, :, -k:])
        case = (kind, shape, world, precision, reg)
        scale = max(1.0, abs(float(want_loss)))
        assert abs(sum(losses) / world - float(want_loss)) < tol * scale, (case, sum(losses) / world, float(want_loss))
        assert abs(sum(losses0) / world - float(want_loss0)) < tol * scale, case
        assert abs(max(maxima) - float(want_max)) < tol * max(1.0, abs(float(want_max))), (case, max(maxima))
        assert abs(sum(means) / world - float(want_mean)) < tol * score_scale, case
        assert rel_err(pg.grad, 3.0 * world * want_dp) < tol, (case, rel_err(pg.grad, 3.0 * world * want_dp))
        assert rel_err(torch.cat(dz), 3.0 * world * want_dz) < tol, (case, rel_err(torch.cat(dz), 3.0 * world * want_dz))


@pytest.mark.gpu
def test_global_negatives_change_nothing_on_one_rank(cpc):
    chans = [16, 24, 24, 24, 32]
    runs = []
    for flag in (False, True):
        torch.manual_seed(0)
        enc = cpc.AudioEncoder({'strides': [5, 4, 2, 2, 2], 'kernel_sizes': [10, 8, 4, 4, 4], 'channel_count': chans,
                                'bias': True})
        model = cpc.AudioPredictiveCodingModel(enc, cpc.AudioGRUModel(32, 16), enc_size=32, ar_size=16,
                                               visible_steps=9, prediction_steps=4).to(DEV)
        trainer = cpc.ContrastiveEstimationTrainer(model=model, dataset=None, device=DEV, regularization=1.0,
                                                   score_function=cpc.softplus_score_function, prediction_steps=4,
                                                   verbose=False, global_negatives=flag)
        x = 0.1 * torch.randn(6, model.item_length, generator=torch.Generator().manual_seed(3))
        loss, mx = trainer.loss_on_batch(x.to(DEV))
        loss.backward()
        runs.append((loss.item(), mx.item(), {n: p.grad.clone() for n, p in model.named_parameters()}))
    (l0, m0, g0), (l1, m1, g1) = runs
    assert abs(l1 - l0) < 1e-6 * abs(l0) and m0 == m1                      # same kernels; fp32 atomics' order only
    for n in g0:
        assert rel_err(g1[n], g0[n]) < 1e-5, n


@pytest.mark.gpu
def test_two_rank_global_negatives(cpc):
    """Two GPUs (skips on one): raw-wave eager and graphed steps against the oracle's global loss and gradients, and
    e24's global loss at the full item length (tests/global_negatives_worker.py)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29751", WORKER, "nccl"],
                         capture_output=True, text=True, timeout=400)
    print(out.stdout[-3000:])
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "RANK_OK 0" in out.stdout and "RANK_OK 1" in out.stdout

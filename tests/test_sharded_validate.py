"""Validation sharded over data-parallel ranks: the partial records of cpc_infonce_validate_ex and their combine (C-ABI
rejections and sizes, host wiring, trainer refusals on CPU), W shards emulated on one B200 against the square
validation kernel and the float64 literal validation block, and ``validate(shard_over_ranks=True)`` on one and on two
GPUs."""
import ctypes
import math
import os
import subprocess
import sys

import pytest
import torch

import cpc_oracle as O

DEV = "cuda:0"
HERE = os.path.dirname(os.path.abspath(__file__))
WORKER = os.path.join(HERE, "sharded_validate_worker.py")


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


def _validate_bytes(b, k, all_steps, pred_batch=None):
    """Validation workspace (lambda = 0): CUDA-core forward scratch, lse, 4 scalars, per-(column tile, row) arg-max;
    rows of pred_batch items (default: the square problem), columns of b items."""
    bp = b if pred_batch is None else pred_batch
    tmr = (64 // k) * k if all_steps else 64
    rows, cols, nprob = (bp * k, b * k, 1) if all_steps else (bp, b, k)
    ncols, nrowtiles, ncoltiles = b * k, -(-rows // tmr), -(-cols // 64)
    ncta, nblk = ncoltiles * nrowtiles * nprob, -(-ncols // 256)
    fwd = 2 * _align(nrowtiles * ncols * 4, 256) + _align(ncols * 4, 256) + _align(ncta * 12, 256) + _align(nblk * 4, 256)
    part = ncoltiles * nprob * rows
    return fwd + _align(ncols * 4, 256) + 256 + 2 * _align(part * 4, 256)


# ---------------------------------------------------------------------------------------------------
# CPU: ABI, sizes, host mirror, trainer refusals
# ---------------------------------------------------------------------------------------------------

def test_validate_ex_and_combine_reject_bad_arguments_before_the_device(built_lib):
    from cpc_b200 import _lib
    lib = _lib.load()
    q = _params(_lib, 4, 3, 8, True)
    fake = ctypes.c_void_p(256)                                     # never dereferenced: every call below is refused
    vex = lambda sh, ws=None, nbytes=0, ptr=fake: lib.cpc_infonce_validate_ex(ptr, ptr, ptr, ctypes.byref(q), sh,  # noqa: E731
                                                                              ws, nbytes, None)
    comb = lambda world, sh, ptr=fake: lib.cpc_infonce_validate_combine(ptr, world, ptr, ctypes.byref(q), sh, None)  # noqa: E731
    # not a rank block: bad shards, the square shard {batch, 0}, pred_batch or offset off the rank grid
    for pred_batch, offset in ((3, 0), (6, 3), (8, -4), (8, 8), (4, 0), (6, 2), (6, 0), (8, 2), (1 << 29, 0)):
        sh = ctypes.byref(_shard(_lib, pred_batch, offset))
        assert vex(sh) == -1 and comb(2, sh) == -1, (pred_batch, offset)
        assert lib.cpc_infonce_validate_partial_bytes(ctypes.byref(q), sh) == 0
        assert lib.cpc_infonce_workspace_bytes_ex(ctypes.byref(q), sh, 2) == 0
    sh = ctypes.byref(_shard(_lib, 12, 8))                          # rank 2 of 3
    need = lib.cpc_infonce_workspace_bytes_ex(ctypes.byref(q), sh, 2)
    assert need > 0
    assert vex(sh, ptr=None) == -7                                  # NULL pointers
    assert vex(sh) == -3 and vex(sh, fake, need - 1) == -3          # no / short workspace
    assert vex(None) == -3                                          # the one-rank record: valid shape, no workspace
    for world in (0, -1, 2, 4):                                     # world < 1, world * batch != pred_batch
        assert comb(world, sh) == -1, world
    assert comb(1, sh) == -1 and comb(2, None) == -1 and comb(0, None) == -1
    assert comb(3, sh, ptr=None) == -7 and comb(1, None, ptr=None) == -7
    q.steps = 100                                                    # K > 64: unsupported, as for every InfoNCE call
    assert vex(sh) == -6 and comb(3, sh) == -6 and lib.cpc_infonce_validate_partial_bytes(ctypes.byref(q), sh) == 0


@pytest.mark.parametrize("all_steps", [True, False])
def test_partial_record_and_workspace_sizes(built_lib, all_steps):
    from cpc_b200 import _lib
    lib = _lib.load()
    for b, k, e, world in ((4, 3, 8, 3), (8, 16, 512, 8), (6, 5, 40, 2), (64, 16, 512, 8)):
        q = _params(_lib, b, k, e, all_steps, _lib.SCORE_LINEAR)
        header = _align(2 * k + 1, 4)
        for r in range(world):
            sh = ctypes.byref(_shard(_lib, world * b, r * b))
            assert lib.cpc_infonce_validate_partial_bytes(ctypes.byref(q), sh) == 4 * (header + 2 * world * b * k)
            # rows of all world * b items against this rank's b columns, on the CUDA-core kernels at every shape
            assert lib.cpc_infonce_workspace_bytes_ex(ctypes.byref(q), sh, 2) == _validate_bytes(b, k, all_steps,
                                                                                                  world * b)
        assert lib.cpc_infonce_validate_partial_bytes(ctypes.byref(q), None) == 4 * (header + 2 * b * k)


@pytest.mark.parametrize("all_steps", [True, False])
def test_square_validation_workspace_unchanged(built_lib, all_steps):
    from cpc_b200 import _lib
    lib = _lib.load()
    for b, k, e in ((4, 3, 8), (64, 16, 512), (33, 5, 100), (200, 12, 64)):
        q = _params(_lib, b, k, e, all_steps)
        assert lib.cpc_infonce_workspace_bytes(ctypes.byref(q), 2) == _validate_bytes(b, k, all_steps)
        assert lib.cpc_infonce_workspace_bytes_ex(ctypes.byref(q), None, 2) == _validate_bytes(b, k, all_steps)


def test_ops_map_validation_shard_and_combine():
    from cpc_b200 import _lib, ops
    pred, z = torch.zeros(12, 5, 40), torch.zeros(6, 40, 7)
    tgt = z[:, :, -5:]
    p = ops._nce_params(pred, tgt, False, "difference", 0.0, "fp32")
    sh = ops._nce_shard(pred, tgt, 6)
    assert (p.batch, p.steps, p.enc, p.score_kind, sh.pred_batch, sh.target_offset) == (6, 5, 40, 2, 12, 6)
    assert (p.tgt_stride_b, p.tgt_stride_e, p.tgt_stride_k) == (280, 7, 1)
    assert ops._nce_flops(p, sh) == 3.0 * 5 * 12 * 6 * 40
    assert "x12" in ops._nce_key("cpc_infonce_validate_ex", p, sh)
    assert ops._nce_shard(pred[:6], tgt, 0) is None                 # one rank: the square record
    recs = torch.zeros(2, 8, dtype=torch.uint8)
    p, sh = ops._nce_combine_args(recs, 6, 5, True)
    assert (p.batch, p.steps, p.all_steps, sh.pred_batch, sh.target_offset) == (6, 5, 1, 12, 0)
    p, sh = ops._nce_combine_args(recs[:1], 6, 5, False)
    assert (p.batch, p.all_steps, sh) == (6, 0, None)
    with pytest.raises(_lib.CpcError):                              # no CPU path
        ops.infonce_validate_shard(pred, tgt, False, "linear", 6)
    with pytest.raises(_lib.CpcError):
        ops.infonce_validate_combine(recs, 6, 5, True)


class _Items(torch.utils.data.Dataset):
    def __init__(self, items):
        self.items = items

    def __len__(self):
        return self.items.shape[0]

    def __getitem__(self, i):
        return self.items[i]

    def get_example_count_per_file(self):
        return [len(self)]


def test_sharded_validate_refusals_come_before_any_collective():
    """With two ranks configured (no process group exists, so a collective would fail differently), each refusal is a
    ValueError raised before anything is gathered or broadcast."""
    from cpc_b200 import trainer as T
    model = torch.nn.Linear(2, 2)
    cases = ((dict(score_function=T.linear_score_function, device="cuda:0"), dict(batch_size=9), "not divisible"),
             (dict(score_function=lambda p, t: T.linear_score_function(p, t), device="cuda:0"), {}, "fused kernels"),
             (dict(score_function=T.softplus_score_function, device="cpu"), {}, "CUDA"),
             (dict(score_function=T.difference_score_function, device=None), {}, "CUDA"))
    for kw, call, msg in cases:
        t = T.ContrastiveEstimationTrainer(model=model, dataset=None, validation_set=_Items(torch.zeros(16, 4)),
                                           verbose=False, **kw)
        t.rank, t.world = 0, 2
        with pytest.raises(ValueError, match=msg):
            t.validate(shard_over_ranks=True, num_workers=0, **dict(dict(batch_size=8), **call))
        assert model.training                                        # refused before model.eval()


# ---------------------------------------------------------------------------------------------------
# GPU: W shards emulated on one device
# ---------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def cpc(built_lib):
    import cpc_b200
    assert cpc_b200._lib.load().cpc_runtime_check() == 0, "device is not a B200 (sm_100)"
    return cpc_b200


@pytest.fixture
def oracle(monkeypatch):
    """cpc_oracle with ``scores_full`` extended by kind='difference', without the (B,K,E,B,K) difference tensor."""
    base = O.scores_full

    def scores_full(pred, targets, kind='linear'):
        if kind != 'difference':
            return base(pred, targets, kind)
        b, k, e = pred.shape
        d = torch.cdist(pred.reshape(b * k, e), targets.permute(0, 2, 1).reshape(-1, e),
                        compute_mode="donot_use_mm_for_euclid_dist") ** 2
        return (1 / d).view(b, k, targets.shape[0], k)
    monkeypatch.setattr(O, "scores_full", scores_full)
    return O


def _literal_validation(oracle, pred, targets, all_steps, kind):
    """The trainer's literal validation block (trainer.validate) on one batch."""
    b, k, _ = pred.shape
    scores = oracle.scores_full(pred, targets, kind)
    n = b * k if all_steps else b
    template = torch.arange(0, n, dtype=torch.long, device=pred.device)
    template = template.view(b, k) if all_steps else template.unsqueeze(1).repeat(1, k)
    if all_steps:
        noise = torch.logsumexp(scores.reshape(-1, b, k), dim=0)
        valid = torch.diagonal(torch.diagonal(scores, dim1=0, dim2=2), dim1=0, dim2=1)
    else:
        scores = torch.diagonal(scores, dim1=1, dim2=3).permute(0, 2, 1).contiguous()
        noise = torch.logsumexp(scores.view(-1, b, k), dim=0)
        valid = torch.diagonal(scores, dim1=0, dim2=2).permute(1, 0)
    losses = -torch.mean(valid - noise, dim=0)
    best = torch.argmax(scores.reshape(b, k, -1), dim=2)
    accuracy = torch.sum(torch.eq(template, best), dim=0).to(pred.dtype) / n
    return losses, accuracy, torch.mean(scores), float(scores.abs().mean())


def _sharded(cpc, pred_all, z_all, k, world, all_steps, kind):
    """W ranks on one device: rank r's record from its targets (strided view) and the concatenated predictions."""
    b = pred_all.shape[0] // world
    records = torch.stack([cpc.ops.infonce_validate_shard(pred_all, z_all[r * b:(r + 1) * b, :, -k:], all_steps, kind,
                                                          target_offset=r * b) for r in range(world)])
    return cpc.ops.infonce_validate_combine(records, b, k, all_steps)


def _inputs(n, k, e, seed, kind):
    gen = torch.Generator().manual_seed(seed)
    z = torch.randn(n, e, k + 2, generator=gen) / math.sqrt(e)                # targets = strided view z[:, :, -k:]
    pred = z[:, :, -k:].permute(0, 2, 1) + 1.5 * torch.randn(n, k, e, generator=gen) / math.sqrt(e)   # partly recognisable
    if kind != "difference":
        pred, z = pred + 0.3, z + 0.3                               # a mean score well away from 0
    return pred, z


def _compare(cpc, oracle, pred, z, k, world, all_steps, kind, case):
    n = pred.shape[0]
    pd, zd = pred.to(DEV), z.to(DEV)
    losses, acc, mean = _sharded(cpc, pd, zd, k, world, all_steps, kind)
    sq_losses, sq_acc, sq_mean = cpc.ops.infonce_validate(pd, zd[:, :, -k:], all_steps, kind)
    want_losses, want_acc, want_mean, score_scale = _literal_validation(oracle, pd.double(), zd[:, :, -k:].double(),
                                                                        all_steps, kind)
    scale = max(1.0, float(want_losses.abs().max()))
    assert float((losses - sq_losses).abs().max()) <= 1e-5 * scale, (case, losses, sq_losses)
    assert torch.equal(acc, sq_acc), (case, acc, sq_acc)
    assert abs(float(mean) - float(sq_mean)) <= 1e-5 * max(abs(float(sq_mean)), score_scale), (case, mean, sq_mean)
    assert float((losses.double() - want_losses).abs().max()) <= 1e-4 * scale, (case, losses, want_losses)
    hits = acc.double().cpu() * (n * k if all_steps else n)
    assert torch.equal(hits.round(), (want_acc.cpu() * (n * k if all_steps else n)).round()), (case, acc, want_acc)
    assert abs(float(mean) - float(want_mean)) <= 1e-4 * max(abs(float(want_mean)), score_scale), (case, mean)
    return acc


# (b, K, E) per shard: K = 5 divides no B_g = W*6 (the per-step scramble moves lse entries across ranks' slots), and
# all-steps rows B_g*K >= 60 span several 60-row tiles; 24 items per shard: per-step rows span several 64-row tiles
# from W = 4 on, all-steps columns two 64-wide tiles
SHAPES = {"k5": (6, 5, 40), "wide": (24, 4, 64)}


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("all_steps", [True, False])
@pytest.mark.parametrize("kind", ["linear", "softplus", "difference"])
def test_shard_records_combine_to_the_whole_batch(cpc, oracle, kind, all_steps, shape, world):
    b, k, e = SHAPES[shape]
    pred, z = _inputs(world * b, k, e, 100 * world + b + k, kind)
    acc = _compare(cpc, oracle, pred, z, k, world, all_steps, kind, (kind, all_steps, shape, world))
    assert float(acc.sum()) > 0.0                                   # the hit counts compared above are not all 0


@pytest.mark.gpu
@pytest.mark.parametrize("all_steps", [True, False])
@pytest.mark.parametrize("kind", ["linear", "softplus", "difference"])
def test_ties_across_ranks_go_to_the_lowest_rank(cpc, oracle, kind, all_steps):
    """Item 5 (rank 1 of 2) repeats the targets of item 1 (rank 0), and item 1's predictions are those targets, while
    item 5's are unrelated.  Every row of item 1 then has its best score twice, at item 1's column (rank 0's record)
    and at item 5's (rank 1's record); the first maximum, rank 0's, wins and the row hits.  A combine that kept the
    last maximum would count a miss for each of these rows, 1/n less accuracy in every slot, and disagree with the
    square kernel and the float64 block."""
    world, b, k, e = 2, 4, 3, 64
    gen = torch.Generator().manual_seed(17)
    z = torch.randn(world * b, e, k + 2, generator=gen) / math.sqrt(e)          # |z|^2 ~ 1, z . z' ~ N(0, 1/64)
    pred = torch.randn(world * b, k, e, generator=gen) / math.sqrt(e)
    z[5] = z[1]
    tgt = z[:, :, -k:]
    pred[1] = tgt[1].t() + (0.05 if kind == "difference" else 0.0)             # D > 0 for the difference kind
    n = world * b * k if all_steps else world * b
    hdr, rows = (2 * k + 1 + 3) // 4 * 4, world * b * k
    pd, td = pred.to(DEV), z.to(DEV)[:, :, -k:]
    # the tie in float64: item 1's rows peak at item 1's and item 5's column alike, and the literal arg-max is item 1's
    s = oracle.scores_full(pd.double(), td.double(), kind)
    s = s.reshape(world * b, k, world * b * k) if all_steps else torch.diagonal(s, dim1=1, dim2=3).permute(0, 2, 1)
    for kk in range(k):
        row = s[1, kk]
        own, dup = (1 * k + kk, 5 * k + kk) if all_steps else (1, 5)
        assert float(row[own]) == float(row[dup]) == float(row.max()) and int(row.argmax()) == own, (kind, kk)
    # each rank's record holds one of the two maxima, with the same value
    recs = [cpc.ops.infonce_validate_shard(pd, td[r * b:(r + 1) * b], all_steps, kind, r * b).cpu() for r in range(2)]
    best = [r.view(torch.float32)[hdr:hdr + rows] for r in recs]
    arg = [r.view(torch.int32)[hdr + rows:hdr + 2 * rows] for r in recs]
    for kk in range(k):
        idx = 1 * k + kk if all_steps else kk * world * b + 1
        assert int(arg[0][idx]) == (1 * k + kk if all_steps else 1), (kk, arg[0][idx])
        assert int(arg[1][idx]) == (5 * k + kk if all_steps else 5), (kk, arg[1][idx])
        assert float(best[0][idx]) == float(best[1][idx])
    # the combine keeps rank 0's: its accuracy equals the square kernel's and the float64 block's, which count the hits
    acc = _compare(cpc, oracle, pred, z, k, world, all_steps, kind, ("ties", kind, all_steps))
    assert all(float(a) >= 1.0 / n - 1e-7 for a in acc), acc                    # item 1's row of every slot hits


@pytest.mark.gpu
@pytest.mark.parametrize("all_steps", [True, False])
@pytest.mark.parametrize("kind", ["linear", "softplus", "difference"])
def test_one_rank_through_the_record_path_matches_infonce_validate(cpc, kind, all_steps):
    b, k, e = 33, 5, 100
    pred, z = _inputs(b, k, e, 5, kind)
    pd, tgt = pred.to(DEV), z.to(DEV)[:, :, -k:]
    rec = cpc.ops.infonce_validate_shard(pd, tgt, all_steps, kind)
    losses, acc, mean = cpc.ops.infonce_validate_combine(rec.unsqueeze(0), b, k, all_steps)
    sq_losses, sq_acc, sq_mean = cpc.ops.infonce_validate(pd, tgt, all_steps, kind)
    assert float((losses - sq_losses).abs().max()) <= 1e-5 * max(1.0, float(sq_losses.abs().max()))
    assert torch.equal(acc, sq_acc)
    assert abs(float(mean) - float(sq_mean)) <= 1e-5 * abs(float(sq_mean))
    again = cpc.ops.infonce_validate_combine(rec.unsqueeze(0).clone(), b, k, all_steps)
    assert all(torch.equal(x, y) for x, y in zip((losses, acc, mean), again))   # the combine is deterministic


@pytest.mark.gpu
def test_shard_over_ranks_changes_nothing_on_one_rank(cpc):
    chans = [16, 24, 24, 24, 32]
    torch.manual_seed(0)
    enc = cpc.AudioEncoder({'strides': [5, 4, 2, 2, 2], 'kernel_sizes': [10, 8, 4, 4, 4], 'channel_count': chans,
                            'bias': True})
    model = cpc.AudioPredictiveCodingModel(enc, cpc.AudioGRUModel(32, 16), enc_size=32, ar_size=16, visible_steps=9,
                                           prediction_steps=4).to(DEV)
    val = _Items(0.1 * torch.randn(16, model.item_length, generator=torch.Generator().manual_seed(3)))
    trainer = cpc.ContrastiveEstimationTrainer(model=model, dataset=None, validation_set=val, device=DEV,
                                               score_function=cpc.softplus_score_function, prediction_steps=4,
                                               verbose=False)
    plain = trainer.validate(batch_size=8, num_workers=0)
    sharded = trainer.validate(batch_size=8, num_workers=0, shard_over_ranks=True)
    for x, y in zip(plain, sharded):
        assert torch.equal(torch.as_tensor(x), torch.as_tensor(y))


@pytest.mark.gpu
def test_two_rank_sharded_validate(cpc):
    """Two GPUs (skips on one): e24 with diverged BatchNorm statistics per rank; validate(shard_over_ranks=True) on both
    ranks against rank 0's validate() of the whole batches (tests/sharded_validate_worker.py)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29753", WORKER],
                         capture_output=True, text=True, timeout=400)
    print(out.stdout[-3000:])
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "RANK_OK 0" in out.stdout and "RANK_OK 1" in out.stdout

"""difference_score_function (S = 1 / |p - z|^2, the reference's third score function) on the fused InfoNCE kernels:
C-ABI and host wiring (CPU), float64 parity, near-coincident pairs, sizes the literal path cannot hold, validation,
non-finite scores and the trainer end to end (GPU)."""
import ctypes
import math

import pytest
import torch

import cpc_oracle as O
from conftest import bn_shadowed_biases, grad_err, rel_err

TOL = 1e-3
DEV = "cuda:0"


def difference_scores(pred, targets):
    """difference_score_function, contrastive_estimation_training.py, restated literally:
    (B,K,E), (B,E,K) -> (B,K,B,K) = 1 / sum_e (pred[d,k,e] - targets[t,e,k'])^2."""
    diff = pred.unsqueeze(3).unsqueeze(4) - targets.permute(1, 0, 2).unsqueeze(0).unsqueeze(1)
    return 1 / torch.sum(diff ** 2, dim=2)


@pytest.fixture
def oracle(monkeypatch):
    """cpc_oracle with ``scores_full`` extended by kind='difference', so that its literal loss block
    (``infonce_loss``, ``infonce_with_grads``) and ``validation_metrics`` evaluate the new kind in float64."""
    base = O.scores_full

    def scores_full(pred, targets, kind='linear'):
        return difference_scores(pred, targets) if kind == 'difference' else base(pred, targets, kind)
    monkeypatch.setattr(O, "scores_full", scores_full)
    return O


@pytest.fixture(scope="module")
def cpc(built_lib):
    import cpc_b200
    assert cpc_b200._lib.load().cpc_runtime_check() == 0, "device is not a B200 (sm_100)"
    return cpc_b200


def _mean_score(scores, all_steps):
    if not all_steps:
        scores = torch.diagonal(scores, dim1=1, dim2=3)
    return scores.mean()


def _close(got, want, tol=TOL):
    return abs(float(got) - float(want)) < tol * max(1.0, abs(float(want)))


# ---------------------------------------------------------------------------------------------------
# CPU: ABI, host mirror, oracle
# ---------------------------------------------------------------------------------------------------

def test_difference_kind_never_takes_the_tensor_path(built_lib):
    """At a size where the linear kind runs on tcgen05 (per-step, 256 candidates, E % 64 == 0), kind 2 is sized for
    the CUDA-core kernels: no backward workspace (per-step, no regulariser) and the CUDA-core forward scratch."""
    from cpc_b200 import _lib
    lib = _lib.load()
    q = _lib.InfoNceParams()
    q.batch, q.steps, q.enc, q.all_steps, q.regularization = 256, 4, 256, 0, 0.0
    q.score_kind = _lib.SCORE_LINEAR
    lin_fwd, lin_bwd = lib.cpc_infonce_workspace_bytes(ctypes.byref(q), 0), lib.cpc_infonce_workspace_bytes(ctypes.byref(q), 1)
    # CUDA-core forward scratch (infonce.cu nce_ws): 4 row tiles x 1024 columns of (max, sum-exp), diagonal,
    # 64 CTAs x (max, sum, reg), 4 combine blocks; each piece aligned to 256 bytes
    core_fwd = 2 * 4 * 1024 * 4 + 1024 * 4 + 768 + 256
    q.score_kind = _lib.SCORE_DIFFERENCE
    assert lin_bwd > 0                                                          # linear: tensor-path operand planes
    assert lib.cpc_infonce_workspace_bytes(ctypes.byref(q), 1) == 0
    assert lib.cpc_infonce_workspace_bytes(ctypes.byref(q), 0) == core_fwd != lin_fwd
    q.all_steps, q.batch, q.steps = 1, 64, 16                                   # e4 / e5 all-steps: 1024 candidates
    assert lib.cpc_infonce_workspace_bytes(ctypes.byref(q), 1) == 0


def test_unknown_score_kind_is_rejected_before_the_device(built_lib):
    from cpc_b200 import _lib
    lib = _lib.load()
    assert _lib.SCORE_DIFFERENCE == 2 and lib.cpc_abi_version() == _lib.ABI_VERSION == 7
    q = _lib.InfoNceParams()
    q.batch, q.steps, q.enc = 4, 3, 8
    for kind in (3, -1):
        q.score_kind = kind
        assert lib.cpc_infonce_workspace_bytes(ctypes.byref(q), 0) == 0
        assert lib.cpc_infonce_fwd(None, None, None, None, ctypes.byref(q), None, 0, None) == -1
        assert lib.cpc_infonce_bwd(None, None, None, None, None, None, ctypes.byref(q), None, 0, None) == -1
        assert lib.cpc_infonce_validate(None, None, None, ctypes.byref(q), None, 0, None) == -1
    q.score_kind = _lib.SCORE_DIFFERENCE                                        # accepted: fails on the null pointers
    assert lib.cpc_infonce_fwd(None, None, None, None, ctypes.byref(q), None, 0, None) == -7


def test_trainer_and_ops_map_difference_score_function():
    from cpc_b200 import _lib, ops, trainer
    assert trainer._FUSED_KINDS[trainer.difference_score_function] == "difference"
    pred, z = torch.zeros(3, 2, 5), torch.zeros(3, 5, 4)
    for precision in ("fp32", "bf16"):
        p = ops._nce_params(pred, z[:, :, -2:], True, "difference", 0.5, precision)
        assert p.score_kind == 2 and p.all_steps == 1 and abs(p.regularization - 0.5) < 1e-7
        lin = ops._nce_params(pred, z[:, :, -2:], True, "linear", 0.5, precision)
        pairs_e = (3 * 2) ** 2 * 5
        assert ops._nce_flops(p) == 3 * pairs_e and ops._nce_bwd_flops(p) == 7 * pairs_e       # + two tile products
        assert ops._nce_flops(lin) == 2 * pairs_e and ops._nce_bwd_flops(lin) == 6 * pairs_e


@pytest.mark.parametrize("all_steps", [False, True])
def test_oracle_difference_loss_is_the_trainers_literal_block(oracle, all_steps):
    """The float64 oracle of the new kind equals the trainer's literal path (difference_score_function +
    reference_loss_from_scores) and, in both modes, the clean cross-entropy over explicit distances."""
    from cpc_b200 import trainer
    b, k, e = 6, 4, 10
    gen = torch.Generator().manual_seed(11)
    pred = torch.randn(b, k, e, generator=gen, dtype=torch.float64)
    z = torch.randn(b, e, k + 2, generator=gen, dtype=torch.float64)
    tgt = z[:, :, -k:]
    for reg in (0.0, 0.3):
        want, want_max = oracle.infonce_loss(pred, tgt, all_steps, 'difference', reg)
        got, got_max = trainer.reference_loss_from_scores(trainer.difference_score_function(pred, tgt), b, k,
                                                          all_steps, reg)
        assert abs(float(got) - float(want)) < 1e-12 and abs(float(got_max) - float(want_max)) < 1e-12
        # clean form: per softmax column, lse over the candidate rows minus the own row
        if all_steps:
            P, Zc = pred.reshape(b * k, e), tgt.permute(0, 2, 1).reshape(b * k, e)
            s = 1 / ((P[:, None, :] - Zc[None, :, :]) ** 2).sum(-1)                # rows (d,k), cols (t,k')
            clean = (torch.logsumexp(s, 0) - torch.diagonal(s)).mean() + reg * (s.view(b, k, -1).mean(1) ** 2).mean()
        else:
            s = 1 / ((pred[:, None, :, :] - tgt.permute(0, 2, 1)[None, :, :, :]) ** 2).sum(-1)   # (d, t, k)
            clean = (torch.logsumexp(s, 0) - torch.diagonal(s).t()).mean() + reg * (s.mean(2) ** 2).mean()
        assert abs(float(clean) - float(want)) < 1e-12


# ---------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------

def _fused(cpc, pred, z, k, all_steps, reg, upstream=3.0, precision=None):
    pg = pred.clone().to(DEV).requires_grad_(True)
    zg = z.clone().to(DEV).requires_grad_(True)
    loss, mx, loss0, mean_s = cpc.ops.infonce(pg, zg[:, :, -k:], all_steps, "difference", reg, precision=precision)
    (upstream * loss).backward()                                 # non-unit upstream gradient
    return loss, mx, loss0, mean_s, pg.grad, zg.grad


def _check_against_oracle(cpc, oracle, pred, z, k, all_steps, reg):
    p64, t64 = pred.to(DEV, torch.float64), z[:, :, -k:].to(DEV, torch.float64)
    want_loss, want_max, want_dp, want_dz = oracle.infonce_with_grads(p64, t64, all_steps, 'difference', reg)
    want_loss0 = oracle.infonce_loss(p64, t64, all_steps, 'difference', 0.0)[0]
    want_mean = _mean_score(oracle.scores_full(p64, t64, 'difference'), all_steps)
    loss, mx, loss0, mean_s, dp, dz = _fused(cpc, pred, z, k, all_steps, reg)
    case = (tuple(pred.shape), all_steps, reg)
    assert _close(loss, want_loss), (case, loss.item(), float(want_loss))
    assert _close(mx, want_max), (case, mx.item(), float(want_max))
    assert _close(loss0, want_loss0), case
    assert abs(mean_s.item() - float(want_mean)) < TOL * abs(float(want_mean)), case
    assert rel_err(dp, 3.0 * want_dp) < TOL, (case, rel_err(dp, 3.0 * want_dp))
    assert rel_err(dz[:, :, -k:], 3.0 * want_dz) < TOL, (case, rel_err(dz[:, :, -k:], 3.0 * want_dz))
    assert float(dz[:, :, :-k].abs().max()) == 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("b,k,e", [(64, 16, 256), (8, 12, 512), (33, 5, 100), (70, 1, 64), (150, 3, 96)])
@pytest.mark.parametrize("all_steps", [False, True])
def test_difference_matches_oracle_with_strided_targets(cpc, oracle, b, k, e, all_steps):
    gen = torch.Generator().manual_seed(b * 1000 + k)
    pred = torch.randn(b, k, e, generator=gen) / math.sqrt(e)
    z = torch.randn(b, e, k + 7, generator=gen) / math.sqrt(e)   # targets = strided view z[:, :, -k:] (audio_model.py:197)
    for reg in (0.0, 0.01, 1.0):
        _check_against_oracle(cpc, oracle, pred, z, k, all_steps, reg)


@pytest.mark.gpu
@pytest.mark.parametrize("b,k,e,all_steps", [(64, 16, 256, True), (150, 3, 96, False)])
def test_difference_near_coincident_pairs(cpc, oracle, b, k, e, all_steps):
    """Half of the predictions sit at their own target plus noise of relative size 1e-2, with |z|^2 ~ 1e3: the near
    pairs have D ~ 0.1 (S ~ 10) against D ~ 2e3 (S ~ 5e-4) for the rest, so (|p|^2 + |z|^2) / D ~ 2e4.  Summing the
    squared differences keeps the 1e-3 bound; the norm expansion |p|^2 + |z|^2 - 2 p.z would not -- about 1e-3 of
    error in fp32 and tens of percent through the 3-pass bf16 tensor-core product."""
    gen = torch.Generator().manual_seed(5 * b + k)
    scale = math.sqrt(1e3 / e)
    z = torch.randn(b, e, k + 5, generator=gen) * scale
    pred = torch.randn(b, k, e, generator=gen) * scale
    near = (torch.arange(b)[:, None] + torch.arange(k)[None, :]) % 2 == 0
    own = z[:, :, -k:].permute(0, 2, 1) + 1e-2 * scale * torch.randn(b, k, e, generator=gen)
    pred[near] = own[near]
    d_near = ((pred - z[:, :, -k:].permute(0, 2, 1)) ** 2).sum(-1)[near]
    assert 0.05 < float(d_near.mean()) < 0.2
    for reg in (0.0, 0.01):
        _check_against_oracle(cpc, oracle, pred, z, k, all_steps, reg)


@pytest.mark.gpu
def test_difference_batch_the_literal_path_cannot_hold(cpc):
    """All-steps B = 512, K = 16, E = 256: R = C = 8192 candidates.  The literal path's (B,K,E,B,K) difference tensor
    would be 68 GB; the fused kernels hold one 64x64 tile.  Checked against a float64 evaluation on the device from
    explicit differences, then at per-step B = 4096, K = 8 against the closed forms (loss ~ 0 when every prediction
    sits at its target, log N when every candidate is equidistant)."""
    b, k, e, reg = 512, 16, 256, 0.01
    gen = torch.Generator(device=DEV).manual_seed(3)
    pred = torch.randn(b, k, e, generator=gen, device=DEV) / math.sqrt(e)
    z = torch.randn(b, e, k + 4, generator=gen, device=DEV) / math.sqrt(e)
    tgt = z[:, :, -k:]
    loss, mx, loss0, mean_s = cpc.ops.infonce(pred, tgt, True, "difference", reg)
    P = pred.reshape(b * k, e).double()
    Zc = tgt.permute(0, 2, 1).reshape(b * k, e).double()                        # column c = t*K + k'
    S = torch.empty(b * k, b * k, dtype=torch.float64, device=DEV)
    for r0 in range(0, b * k, 512):
        D = torch.cdist(P[r0:r0 + 512], Zc, compute_mode="donot_use_mm_for_euclid_dist") ** 2
        S[r0:r0 + 512] = 1 / D
    want0 = (torch.logsumexp(S, dim=0) - torch.diagonal(S)).mean()
    want = want0 + reg * (S.view(b, k, b * k).mean(1) ** 2).mean()
    assert _close(loss, want) and _close(loss0, want0), (loss.item(), float(want))
    assert _close(mx, S.max()) and abs(mean_s.item() - float(S.mean())) < TOL * float(S.mean())
    del S
    b, k, e = 4096, 8, 128
    z = torch.randn(b, e, k, generator=gen, device=DEV)
    zn = z / z.norm(dim=1, keepdim=True)
    pred = zn.permute(0, 2, 1).contiguous() + 1e-3 * torch.randn(b, k, e, generator=gen, device=DEV)
    loss, _, _, _ = cpc.ops.infonce(pred, zn, False, "difference", 0.0)
    assert loss.item() < 1e-3
    loss, mx, _, _ = cpc.ops.infonce(torch.zeros_like(pred), zn, False, "difference", 0.0)     # S = 1 / |z|^2 = 1
    assert abs(loss.item() - math.log(b)) < 1e-5 and abs(mx.item() - 1.0) < 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("b,k,e", [(33, 5, 100), (16, 12, 64)])
@pytest.mark.parametrize("all_steps", [False, True])
def test_difference_validate_matches_oracle(cpc, oracle, b, k, e, all_steps):
    gen = torch.Generator().manual_seed(7 * b + k)
    z = torch.randn(b, e, k + 2, generator=gen) / math.sqrt(e)
    tgt = z[:, :, -k:]
    pred = tgt.permute(0, 2, 1) + 1.5 * torch.randn(b, k, e, generator=gen) / math.sqrt(e)    # partly recognisable
    losses, acc, score = cpc.ops.infonce_validate(pred.to(DEV), z.to(DEV)[:, :, -k:], all_steps, "difference")
    want = oracle.validation_metrics(pred.double(), tgt.double(), all_steps, 'difference')
    scale = max(1.0, float(want[0].abs().max()))
    assert float((losses.cpu().double() - want[0]).abs().max()) < TOL * scale
    n = b * k if all_steps else b
    assert torch.equal((acc.cpu().double() * n).round(), (want[1] * n).round()), (acc, want[1])   # hit counts: exact
    assert float(want[1].sum()) > 0.0
    assert abs(float(score) - float(want[2])) < TOL * abs(float(want[2]))


@pytest.mark.gpu
@pytest.mark.parametrize("all_steps", [False, True])
def test_difference_prediction_equal_to_target_gives_non_finite_loss(cpc, all_steps):
    from cpc_b200 import trainer as T
    b, k, e = 6, 3, 16
    gen = torch.Generator().manual_seed(2)
    pred = torch.randn(b, k, e, generator=gen)
    tgt = torch.randn(b, e, k, generator=gen)
    pred[2, 1] = tgt[2, :, 1]                                                   # D = 0, S = +inf
    loss, mx, _, _ = cpc.ops.infonce(pred.to(DEV), tgt.to(DEV), all_steps, "difference", 0.01)
    literal, _ = T.reference_loss_from_scores(T.difference_score_function(pred.to(DEV), tgt.to(DEV)), b, k, all_steps,
                                              0.01)
    assert not math.isfinite(literal.item()) and not math.isfinite(loss.item())
    assert mx.item() == math.inf


class _Items(torch.utils.data.Dataset):
    def __init__(self, items):
        self.items = items

    def __len__(self):
        return self.items.shape[0]

    def __getitem__(self, i):
        return self.items[i]

    def get_example_count_per_file(self):
        return [len(self)]


class _CoincidentModel(torch.nn.Module):
    """Returns fixed predictions and targets; prediction (0, 0) equals its own target."""

    def __init__(self, b, k, e):
        super().__init__()
        gen = torch.Generator().manual_seed(4)
        self.pred = torch.nn.Parameter(torch.randn(b, k, e, generator=gen))
        t = torch.randn(b, e, k, generator=gen)
        t[0, :, 0] = self.pred.detach()[0, 0]
        self.register_buffer("targets", t)

    def forward(self, x):
        return self.pred + 0.0 * x.mean(), self.targets, None, None


@pytest.mark.gpu
def test_difference_train_returns_before_the_optimizer_step_on_a_non_finite_loss(cpc):
    b, k, e = 4, 3, 8
    model = _CoincidentModel(b, k, e).to(DEV)
    before = model.pred.detach().clone()
    trainer = cpc.ContrastiveEstimationTrainer(model=model, dataset=_Items(torch.randn(b, 32)), device=DEV,
                                               optimizer=torch.optim.SGD, score_function=cpc.difference_score_function,
                                               score_over_all_timesteps=True, regularization=0.01,
                                               prediction_steps=k, verbose=False)
    trainer.train(batch_size=b, epochs=1, lr=0.1, num_workers=0, max_steps=1)
    assert math.isnan(trainer.last_loss)
    assert torch.equal(model.pred.detach(), before) and model.pred.grad is None


@pytest.mark.gpu
def test_difference_trainer_end_to_end_matches_literal_path(cpc):
    """experiment('e24') with score_function=difference_score_function, 8 items at the full item length: the fused
    trainer against the same trainer given a wrapper of the function (not recognised, so it runs the literal block).
    The network before the score is the same code on both sides, so the ReLU gates coincide and every parameter
    gradient is comparable; validate() on an in-memory set and one CUDA-graph capture of the fused step as well."""
    exp = cpc.configs.experiment("e24")
    tc = exp["training_config"]
    dev = torch.device(DEV)

    def make(score_function):
        torch.manual_seed(0)
        model, pre, _ = cpc.configs.setup_model(exp["cqt_config"], exp["encoder_config"], exp["ar_model_config"], tc,
                                                device=dev)
        trainer = cpc.ContrastiveEstimationTrainer(model=model, dataset=None, device=dev, regularization=0.01,
                                                   score_over_all_timesteps=tc["score_over_all_timesteps"],
                                                   score_function=score_function, preprocessing=pre,
                                                   prediction_steps=tc["prediction_steps"], verbose=False)
        return model, trainer

    literal_fn = lambda p, t: cpc.difference_score_function(p, t)              # noqa: E731 -- not in _FUSED_KINDS
    (m_f, t_f), (m_l, t_l) = make(cpc.difference_score_function), make(literal_fn)
    for (n, p), (_, q) in zip(m_f.named_parameters(), m_l.named_parameters()):
        assert torch.equal(p, q), n
    gen = torch.Generator().manual_seed(2)
    x = 0.1 * torch.randn(8, m_f.item_length, generator=gen)
    # validation first, while the two models are identical
    val = _Items(0.1 * torch.randn(8, m_f.item_length, generator=gen))
    t_f.validation_set = t_l.validation_set = val
    vf, vl = t_f.validate(batch_size=8, num_workers=0), t_l.validate(batch_size=8, num_workers=0)
    assert float((vf[0] - vl[0]).abs().max()) < TOL * max(1.0, float(vl[0].abs().max()))
    assert torch.equal(vf[1], vl[1]) and abs(vf[2] - vl[2]) < TOL * abs(vl[2])
    noise_only = bn_shadowed_biases(m_f.state_dict().keys())
    runs = {}
    for name, model, trainer in (("fused", m_f, t_f), ("literal", m_l, t_l)):
        model.train()
        opt = torch.optim.SGD(model.parameters(), lr=1e-4)
        out = []
        for _ in range(2):
            loss, mx = trainer.loss_on_batch(x.to(DEV))
            opt.zero_grad(set_to_none=True)
            loss.backward()
            out.append((loss.item(), mx.item(), {n: p.grad.clone() for n, p in model.named_parameters()}))
            opt.step()
        runs[name] = out
    for (lf, mf, gf), (ll, ml, gl) in zip(runs["fused"], runs["literal"]):
        assert math.isfinite(lf) and abs(lf - ll) < TOL * max(1.0, abs(ll)), (lf, ll)
        assert abs(mf - ml) < TOL * max(1.0, abs(ml)), (mf, ml)
        for n in gl:
            if n not in noise_only:
                assert grad_err(gf[n], gl[n]) < TOL, (n, grad_err(gf[n], gl[n]))
    m_g, t_g = make(cpc.difference_score_function)
    m_g.train()
    step = cpc.GraphedTrainStep(t_g, torch.optim.Adam(m_g.parameters(), lr=1e-4, capturable=True),
                                (8, m_g.item_length), warmup=2)
    graphed, _ = step(x.pin_memory())
    assert abs(graphed.item() - runs["fused"][0][0]) < 1e-4 * max(1.0, abs(runs["fused"][0][0]))


@pytest.mark.gpu
@pytest.mark.parametrize("b,k,e,all_steps,reg", [(33, 5, 100, False, 0.0), (8, 8, 64, True, 0.01),
                                                 (150, 3, 96, False, 0.01)])
def test_difference_bf16_operand_mode_is_bit_identical(cpc, b, k, e, all_steps, reg):
    """The difference kind always runs on the fp32 CUDA-core kernels, so precision="bf16" changes nothing.  At one tile
    per problem (the first two cases) every gradient entry receives exactly one atomic add and the results are compared
    bit for bit; with several tiles the atomics' order varies between ANY two runs, so the third case is held to 1e-6."""
    gen = torch.Generator().manual_seed(b + k)
    pred = torch.randn(b, k, e, generator=gen) / math.sqrt(e)
    z = torch.randn(b, e, k + 1, generator=gen) / math.sqrt(e)
    a = _fused(cpc, pred, z, k, all_steps, reg, precision="fp32")
    c = _fused(cpc, pred, z, k, all_steps, reg, precision="bf16")
    if b * (k if all_steps else 1) <= 64:
        for x, y in zip(a, c):
            assert torch.equal(x, y)
    else:
        for x, y in zip(a, c):
            assert rel_err(x, y) < 1e-6

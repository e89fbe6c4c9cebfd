"""train(cuda_graph=True): one captured CUDA graph per step, with the reference's NaN stop decided on the device.

CPU: ``cpc_adam_step_ex`` is exported and rejects what ``cpc_adam_step`` rejects, before the device is touched; the
refusals of ``train(cuda_graph=True)`` come before any collective; ``GraphedTrainStep(stop_on_nan=True)`` needs
``cpc_b200.optim.Adam``.
One GPU: the guarded Adam bit for bit against the unguarded one, eagerly and inside a replayed graph; graphed against
eager ``train()`` on WAV folders (both feeds, a scalogram and a raw-wave model); a NaN stop built deterministically;
hooks and the loader thread cleaned up on every exit.  Two GPUs (skips on one): tests/graphed_train_worker.py.
"""
import ctypes
import os
import random
import subprocess
import sys

import pytest
import torch

from conftest import bn_shadowed_biases
from test_device_loader import _loader_threads, _refusing_trainer, make_folder

DEV = "cuda:0"
HERE = os.path.dirname(os.path.abspath(__file__))
WORKER = os.path.join(HERE, "graphed_train_worker.py")


# ---------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------

def test_adam_step_ex_rejects_what_adam_step_rejects(built_lib):
    from cpc_b200 import _lib
    lib = _lib.load()
    assert hasattr(ctypes.CDLL(built_lib), "cpc_adam_step_ex")
    state = (ctypes.c_float * 4)()
    skip = (ctypes.c_float * 1)()
    ptrs = (ctypes.c_void_p * 1)(4096)
    odd = (ctypes.c_void_p * 1)(4098)
    nulls = (ctypes.c_void_p * 1)(0)

    def cases():
        a = _lib.AdamParams(1e-3, 0.9, 0.999, 1e-8, 0.0, 1.0, 0)
        yield (0, None, None, None, None, None, None, a), -7                          # no step counter
        yield (1, None, None, None, None, (ctypes.c_int64 * 1)(4), state, a), -7       # no pointer tables
        yield (1, nulls, ptrs, ptrs, ptrs, (ctypes.c_int64 * 1)(4), state, a), -7      # a NULL tensor
        yield (1, odd, ptrs, ptrs, ptrs, (ctypes.c_int64 * 1)(4), state, a), -2        # not 4-byte aligned
        yield (1, ptrs, ptrs, ptrs, ptrs, (ctypes.c_int64 * 1)(-1), state, a), -1      # negative numel
        yield (-1, None, None, None, None, None, state, a), -1                         # negative count
        for field, value in (("beta1", 1.0), ("beta2", 1.5), ("eps", -1.0)):
            bad = _lib.AdamParams(1e-3, 0.9, 0.999, 1e-8, 0.0, 1.0, 0)
            setattr(bad, field, value)
            yield (0, None, None, None, None, None, state, bad), -1
    for (n, p, g, m, v, numel, st, a), want in cases():
        plain = lib.cpc_adam_step(n, p, g, m, v, numel, st, ctypes.byref(a), None)
        assert plain == want
        for flag in (None, skip):                                   # NULL skip: "always update", accepted
            assert lib.cpc_adam_step_ex(n, p, g, m, v, numel, st, flag, ctypes.byref(a), None) == want


@pytest.mark.parametrize("world", [1, 2])
def test_train_cuda_graph_refusals_come_before_any_collective(tmp_path, world):
    """With two ranks configured but no process group, a collective would fail with a different error: each refusal
    is a ValueError raised before anything is broadcast."""
    for device in ("cpu", None):
        t = _refusing_trainer(tmp_path, device, world=world)
        with pytest.raises(ValueError, match="CUDA"):
            t.train(batch_size=2, epochs=1, cuda_graph=True)
    t = _refusing_trainer(tmp_path, "cuda:0", world=world)
    t.wasserstein_gradient_penalty = True
    with pytest.raises(ValueError, match="gradient penalty"):
        t.train(batch_size=2, epochs=1, cuda_graph=True)
    t = _refusing_trainer(tmp_path, "cuda:0", world=world)
    with pytest.raises(ValueError, match="profile"):
        t.train(batch_size=2, epochs=1, cuda_graph=True, profile=True)
    # the model's parameters are on the CPU, so make_optimizer keeps torch.optim.Adam; and any other class
    for cls in (torch.optim.Adam, torch.optim.SGD):
        t = _refusing_trainer(tmp_path, "cuda:0", world=world)
        t.optimizer = cls
        with pytest.raises(ValueError, match="cpc_b200.optim.Adam"):
            t.train(batch_size=2, epochs=1, cuda_graph=True, device_loading=True)
        assert t.model.training


def test_graphed_step_stop_on_nan_needs_cpc_adam(tmp_path):
    from cpc_b200 import trainer as T
    t = _refusing_trainer(tmp_path, "cpu")
    with pytest.raises(ValueError, match="cpc_b200.optim.Adam"):
        T.GraphedTrainStep(t, torch.optim.Adam(t.model.parameters()), (2, 8), stop_on_nan=True)


# ---------------------------------------------------------------------------------------------------
# One GPU: the guarded Adam
# ---------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def cpc(built_lib):
    import cpc_b200
    assert cpc_b200._lib.load().cpc_runtime_check() == 0, "device is not a B200 (sm_100)"
    return cpc_b200


SHAPES = [(512, 256, 5), (4097,), (1,), (3, 3), (8192,)] + [(17 + i,) for i in range(55)]   # 60 tensors: 2 launches


def _adam_pair(cpc, weight_decay, maximize, seed=3):
    gen = torch.Generator().manual_seed(seed)
    base = [torch.randn(s, generator=gen) for s in SHAPES]
    sets = [[b.clone().to(DEV).requires_grad_(True) for b in base] for _ in range(2)]
    opts = [cpc.optim.Adam(ps, lr=3e-3, weight_decay=weight_decay, maximize=maximize) for ps in sets]
    return sets, opts, gen


def _state(ps, opt):
    out = [p.detach().clone() for p in ps]
    for p in ps:
        st = opt.state.get(p, {})
        out += [st[k].detach().clone() for k in ("exp_avg", "exp_avg_sq") if k in st]
    counter = opt.param_groups[0].get('_step_state')
    out.append(counter[0].clone() if counter is not None else torch.zeros((), device=DEV))
    return out


def _assert_equal(a, b):
    assert len(a) == len(b)
    for i, (x, y) in enumerate(zip(a, b)):
        assert torch.equal(x, y), i


@pytest.mark.gpu
@pytest.mark.parametrize("weight_decay,maximize,grad_scale", [(0.0, False, 1.0), (0.01, False, 1.0),
                                                               (0.0, True, 1.0), (0.0, False, 0.25)])
def test_guarded_adam_is_bit_identical_or_a_no_op(cpc, weight_decay, maximize, grad_scale):
    (pa, pb), (oa, ob), gen = _adam_pair(cpc, weight_decay, maximize)
    zero, one = torch.zeros(1, device=DEV), torch.ones(1, device=DEV)
    for step in range(4):
        for a, b in zip(pa, pb):
            g = torch.randn(a.shape, generator=gen).to(DEV) * (10.0 ** (step % 3 - 2))
            a.grad, b.grad = g.clone(), g.clone()
        oa.step(grad_scale=grad_scale)
        ob.step(grad_scale=grad_scale, skip_if=zero)
        _assert_equal(_state(pa, oa), _state(pb, ob))
        before = _state(pb, ob)
        ob.step(grad_scale=grad_scale, skip_if=one)                  # changes nothing, not even the step count
        _assert_equal(before, _state(pb, ob))
    assert float(ob.state_dict()['state'][0]['step']) == 4.0


@pytest.mark.gpu
@pytest.mark.parametrize("weight_decay,maximize,grad_scale", [(0.0, False, 1.0), (0.01, True, 0.5)])
def test_guarded_adam_decides_per_replay_of_a_graph(cpc, weight_decay, maximize, grad_scale):
    """A captured guarded step replayed with the flag at 0, 1, 0 equals two eager updates."""
    (pa, pb), (oa, ob), gen = _adam_pair(cpc, weight_decay, maximize, seed=7)
    grads = [[torch.randn(s, generator=gen).to(DEV) for s in SHAPES] for _ in range(3)]
    flag = torch.ones(1, device=DEV)
    for b in pb:
        b.grad = torch.zeros_like(b)
    ob.step(grad_scale=grad_scale, skip_if=flag)                     # creates the state outside the capture; no-op
    _assert_equal([p.detach().clone() for p in pa], [p.detach().clone() for p in pb])
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        ob.step(grad_scale=grad_scale, skip_if=flag)
    for i, (gs, f) in enumerate(zip(grads, (0.0, 1.0, 0.0))):
        for b, g in zip(pb, gs):
            b.grad.copy_(g)
        flag.fill_(f)
        graph.replay()
        if f == 0.0:
            for a, g in zip(pa, gs):
                a.grad = g.clone()
            oa.step(grad_scale=grad_scale)
        torch.cuda.synchronize()
        _assert_equal(_state(pa, oa), _state(pb, ob))
    assert float(ob.state_dict()['state'][0]['step']) == 2.0


# ---------------------------------------------------------------------------------------------------
# One GPU: train(cuda_graph=True) against train()
# ---------------------------------------------------------------------------------------------------

class _Meter:
    def __init__(self):
        self.values = []

    def update(self, v):
        self.values.append(v)


class RecordingLogger:
    """The logger interface train() calls per step; ``on_log(step)`` runs after each step's update."""

    def __init__(self, on_log=None):
        self.loss_meter, self.score_meter, self.steps, self.on_log = _Meter(), _Meter(), [], on_log

    def log(self, step):
        self.steps.append(step)
        if self.on_log is not None:
            self.on_log(step)


def _scalogram_model(cpc):
    from test_gpu_parity import small_resnet_cfg
    cfg = small_resnet_cfg()
    cfg['blocks'][2] = dict(cfg['blocks'][2], kernel_size_1=(30, 2), pooling_1=1, ceil_pooling=False)
    cfg['blocks'][1] = dict(cfg['blocks'][1], kernel_size_2=(35, 1))
    pre = cpc.PreprocessingModule(dict(cpc.cqt_default_dict), phase=True)
    enc = cpc.ScalogramResidualEncoder(cfg, preprocessing_module=pre)
    ar = cpc.ConvolutionalArModel({'kernel_sizes': [3, 3], 'channel_count': [24, 16, 16], 'stride': [1, 1],
                                   'pooling': [1, 2], 'bias': True, 'batch_norm': True, 'residual': False,
                                   'activation_register': None})
    model = cpc.AudioPredictiveCodingModel(enc, ar, enc_size=24, ar_size=16, visible_steps=10, prediction_steps=3)
    return model.to(DEV), pre.to(DEV), dict(regularization=0.1, score_over_all_timesteps=True,
                                            score_function=cpc.linear_score_function, prediction_steps=3)


def _raw_model(cpc):
    enc = cpc.AudioEncoder({'strides': [5, 4, 2, 2, 2], 'kernel_sizes': [10, 8, 4, 4, 4],
                            'channel_count': [16, 24, 24, 24, 32], 'bias': True})
    model = cpc.AudioPredictiveCodingModel(enc, cpc.AudioGRUModel(32, 16), enc_size=32, ar_size=16, visible_steps=9,
                                           prediction_steps=4)
    return model.to(DEV), None, dict(score_function=cpc.softplus_score_function, prediction_steps=4)


def _setup(cpc, root, kind, logger=None):
    """Model, trainer (and the optimizer train() makes, once it has made it) on a synthetic 16-bit WAV folder."""
    from cpc_b200.audio_dataset import AudioDataset
    torch.manual_seed(5)
    model, pre, kw = (_scalogram_model if kind == "scalogram" else _raw_model)(cpc)
    n = model.item_length
    root = root / kind                                             # files sized for this model's item length
    if not (root / "f00.wav").exists():
        make_folder(root, [3 * n + 17, n // 2, n // 3 + 5, 4 * n, 2 * n + 1, n + 3], 1, 2, seed=40)
    ds = AudioDataset(root, item_length=n, unique_length=n * 3 // 4)
    trainer = cpc.ContrastiveEstimationTrainer(model=model, dataset=ds, device=DEV, preprocessing=pre, logger=logger,
                                               verbose=False, **kw)
    made = []
    plain = trainer.make_optimizer

    def recording(lr, **kwargs):
        made.append(plain(lr, **kwargs))
        return made[-1]
    trainer.make_optimizer = recording
    return trainer, made


def _adam_state(opt):
    """Every parameter, both moments of every parameter that has them, and the device step count."""
    ps = [p for g in opt.param_groups for p in g['params']]
    return ([p.detach().clone() for p in ps] + [opt.state[p][k].detach().clone() for p in ps if p in opt.state
                                                for k in ("exp_avg", "exp_avg_sq")]
            + [opt.param_groups[0]['_step_state'][0].clone()])


def _run(cpc, root, kind, cuda_graph, device_loading, **train_kw):
    logger = RecordingLogger()
    trainer, made = _setup(cpc, root, kind, logger)
    random.seed(123)                                               # FileBatchSampler draws from `random`
    trainer.train(batch_size=4, lr=1e-3, num_workers=0, device_loading=device_loading, cuda_graph=cuda_graph,
                  **train_kw)
    assert not _loader_threads()
    return trainer, made[0], logger


def _assert_close_parameters(m_eager, m_graph, steps, lr=1e-3):
    """test_gpu_parity.test_cuda_graph_step_reproduces_eager_steps's bound: conv biases in front of a BatchNorm carry
    only rounding noise; elsewhere 1e-4 relative plus 2 % of the lr-sized steps taken."""
    noise_only = bn_shadowed_biases(m_eager.state_dict().keys())
    for (n, p), (_, q) in zip(m_eager.named_parameters(), m_graph.named_parameters()):
        if n not in noise_only:
            slack = 1e-4 * float(p.detach().abs().max()) + 0.02 * steps * lr
            assert float((q.detach() - p.detach()).abs().max()) < slack, n


@pytest.mark.gpu
@pytest.mark.parametrize("device_loading", [False, True])
@pytest.mark.parametrize("kind,train_kw", [("scalogram", dict(epochs=3, max_steps=7, continue_training_at_step=3)),
                                           ("raw", dict(epochs=2, continue_training_at_step=2))])
def test_graphed_train_matches_eager_train(cpc, tmp_path, kind, train_kw, device_loading):
    root = tmp_path / "wav"
    t_e, o_e, l_e = _run(cpc, root, kind, False, device_loading, **train_kw)
    t_g, o_g, l_g = _run(cpc, root, kind, True, device_loading, **train_kw)
    start = train_kw["continue_training_at_step"]
    assert isinstance(o_g, cpc.optim.Adam)
    assert l_g.steps == l_e.steps and l_e.steps[0] == start and len(l_e.steps) >= 4, (l_e.steps, l_g.steps)
    if "max_steps" in train_kw:
        assert l_e.steps[-1] == train_kw["max_steps"] - 1
    assert t_g.training_step == t_e.training_step == start + len(l_e.steps)
    steps = len(l_e.steps)
    assert float(o_g.state_dict()['state'][0]['step']) == float(o_e.state_dict()['state'][0]['step']) == steps
    for a, b in zip(l_e.loss_meter.values, l_g.loss_meter.values):
        assert abs(a - b) <= 1e-4 * max(1.0, abs(a)), (l_e.loss_meter.values, l_g.loss_meter.values)
    assert t_g.last_loss == l_g.loss_meter.values[-1] and t_g.last_max_score == l_g.score_meter.values[-1]
    _assert_close_parameters(t_e.model, t_g.model, steps)


def _poisoned_run(cpc, root, cuda_graph, stop_at, device_loading=True):
    """predicted_z is multiplied by a device scalar that the logger sets to NaN at step stop_at - 1, after taking a
    snapshot of weights and Adam state; BatchNorm statistics stay finite."""
    poison = torch.ones((), device=DEV)
    snap = {}
    holder = {}

    def on_log(step):
        if step == stop_at - 1:
            snap["state"] = _adam_state(holder["opt"][0])
            poison.fill_(float("nan"))
    logger = RecordingLogger(on_log)
    trainer, made = _setup(cpc, root, "scalogram", logger)
    holder["opt"] = made
    trainer.model.register_forward_hook(lambda mod, inp, out: (out[0] * poison,) + tuple(out[1:]))
    random.seed(123)
    trainer.train(batch_size=4, epochs=3, lr=1e-3, num_workers=0, device_loading=device_loading,
                  cuda_graph=cuda_graph)
    assert not _loader_threads()
    return trainer, made[0], logger, snap["state"]


@pytest.mark.gpu
def test_graphed_train_stops_on_nan_like_the_eager_loop(cpc, tmp_path, capsys):
    root = tmp_path / "wav"
    stop_at = 3
    t_e, o_e, l_e, snap_e = _poisoned_run(cpc, root, False, stop_at)
    out_e = capsys.readouterr().out
    t_g, o_g, l_g, snap_g = _poisoned_run(cpc, root, True, stop_at)
    out_g = capsys.readouterr().out
    for t, l, out in ((t_e, l_e, out_e), (t_g, l_g, out_g)):
        assert t.training_step == stop_at and l.steps == list(range(stop_at))
        assert t.last_loss != t.last_loss                             # NaN
        assert "nan loss\nreturned with nan loss at step %d\n" % stop_at in out
    _assert_equal(snap_g, _adam_state(o_g))                          # the NaN step changed nothing the optimizer owns
    _assert_equal(snap_e, _adam_state(o_e))
    assert float(o_g.state_dict()['state'][0]['step']) == stop_at
    # the NaN step's forward updated the running statistics on both paths (its batch is the same)
    bufs_e, bufs_g = dict(t_e.model.named_buffers()), dict(t_g.model.named_buffers())
    for name, b in bufs_e.items():
        g = bufs_g[name]
        assert bool(torch.isfinite(g.float()).all()), name
        if b.dtype.is_floating_point:
            assert float((g - b).abs().max()) <= 1e-3 * max(1.0, float(b.abs().max())), name
        else:
            assert torch.equal(g, b), name


def _hooks_left(model):
    return sum(len(getattr(p, "_post_accumulate_grad_hooks", None) or {}) for p in model.parameters())


@pytest.mark.gpu
def test_graphed_train_cleans_up_on_every_exit(cpc, tmp_path):
    root = tmp_path / "wav"
    # normal end (max_steps) and NaN stop
    t, _, _ = _run(cpc, root, "raw", True, True, epochs=1, max_steps=2)
    assert t.training_step == 2 and _hooks_left(t.model) == 0 and not _loader_threads()
    t, _, _, _ = _poisoned_run(cpc, root, True, 2)
    assert _hooks_left(t.model) == 0 and not _loader_threads()

    # an exception raised by the dataset mid-epoch (DataLoader feed) ...
    trainer, _ = _setup(cpc, root, "raw")
    calls = {"n": 0}
    plain = trainer.dataset.__class__.__getitem__

    class Failing(trainer.dataset.__class__):
        def __getitem__(self, i):
            calls["n"] += 1
            if calls["n"] > 9:
                raise RuntimeError("unreadable item")
            return plain(self, i)
    trainer.dataset.__class__ = Failing
    random.seed(123)
    with pytest.raises(RuntimeError, match="unreadable item"):
        trainer.train(batch_size=4, epochs=2, lr=1e-3, num_workers=0, cuda_graph=True)
    assert 1 <= trainer.training_step and _hooks_left(trainer.model) == 0

    # ... and one raised mid-epoch with the device loader's thread running
    def failing_log(step):
        if step == 1:
            raise RuntimeError("logger failed")
    trainer, _ = _setup(cpc, root, "raw", RecordingLogger(failing_log))
    random.seed(123)
    with pytest.raises(RuntimeError, match="logger failed"):
        trainer.train(batch_size=4, epochs=2, lr=1e-3, device_loading=True, cuda_graph=True)
    assert _hooks_left(trainer.model) == 0 and not _loader_threads()


# ---------------------------------------------------------------------------------------------------
# Two GPUs
# ---------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_two_rank_graphed_train(cpc):
    """Two GPUs (skips on one): tests/graphed_train_worker.py."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29761", WORKER],
                         capture_output=True, text=True, timeout=600)
    print(out.stdout[-3000:])
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "RANK_OK 0" in out.stdout and "RANK_OK 1" in out.stdout

"""GPU parity tests (-m gpu): the CUDA path, called through the Python host mirror -> ctypes -> C-ABI,
against (a) the golden vectors the unmodified reference produced and (b) the CPU oracle on fresh seeded
inputs.  Tolerances follow the north star: 1e-3 relative (norm-wise) in fp32 mode for CQT magnitudes,
encoder outputs, InfoNCE loss and gradients; sampler indices are covered bit-exactly on CPU."""
import copy
import json
import math
import random

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import cpc_oracle as O
from conftest import bn_shadowed_biases, grad_err, load_golden, rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-3          # north-star fp32 tolerance
DEV = "cuda:0"


@pytest.fixture(scope="module")
def cpc(built_lib):
    import cpc_b200
    assert cpc_b200._lib.load().cpc_runtime_check() == 0, "device is not a B200 (sm_100)"
    return cpc_b200


def phase_err_fraction(a, b, scale, tol=1e-3):
    """fraction of phase-difference entries whose circular distance exceeds tol (scale: (F,) per-bin factor)."""
    a = torch.as_tensor(a, dtype=torch.float64).cpu()
    b = torch.as_tensor(b, dtype=torch.float64).cpu()
    s = torch.as_tensor(scale, dtype=torch.float64).view(1, -1, 1)
    d = (a - b) / s
    d = torch.remainder(d + math.pi, 2 * math.pi) - math.pi
    return float((d.abs() > tol).double().mean())


# ---------------------------------------------------------------------------------------------------
# CQT front end
# ---------------------------------------------------------------------------------------------------

def test_cqt_complex_and_scalograms_match_reference_golden(cpc):
    g = load_golden("cqt.npz")
    x = torch.from_numpy(g["x"]).to(DEV)
    cqt = cpc.CQT(sr=16000, fmin=30, n_bins=256, bins_per_octave=32, filter_scale=0.5, hop_length=128).to(DEV)
    z = cqt(x)
    assert tuple(z.shape) == g["complex"].shape
    assert rel_err(z, g["complex"]) < TOL
    d = dict(cpc.cqt_default_dict)
    y = cpc.PreprocessingModule(d, phase=False).to(DEV)(x)
    assert y.grad_fn is None and not y.requires_grad            # must be an autograd leaf (trainer sets requires_grad)
    assert rel_err(y, g["logpow"]) < TOL                        # includes exact -inf on the silent stretch
    pre = cpc.PreprocessingModule(d, phase=True).to(DEV)
    y = pre(x)
    assert tuple(y.shape) == g["logpow_phase"].shape
    assert rel_err(y[:, 0], g["logpow_phase"][:, 0]) < TOL
    scale = pre.phase_diff.scaling.reshape(-1).cpu()
    assert phase_err_fraction(y[:, 1], g["logpow_phase"][:, 1], scale) < 2e-3
    y = cpc.PreprocessingModule(d, phase=False, offset_zero=True, output_power=2., pooling=[1, 2], scaling=10.).to(DEV)(x)
    assert rel_err(y, g["offset_pool_power"]) < TOL
    y = cpc.PreprocessingModule(d, phase=True, offset_zero=True, pooling=[1, 2]).to(DEV)(x)
    assert tuple(y.shape) == g["phase_offset_pool"].shape
    assert rel_err(y[:, 0], g["phase_offset_pool"][:, 0]) < TOL
    cqt2 = cpc.CQT(sr=8000, fmin=55, n_bins=120, bins_per_octave=24, filter_scale=1., hop_length=64).to(DEV)
    assert rel_err(cqt2(torch.from_numpy(g["x2"]).to(DEV)), g["complex2"]) < TOL


def test_high_res_cqt_matches_reference_golden(cpc):
    """The filterbank of experiments e27 ... e32 (cqt_high_res_dict: 44.1 kHz, 292 bins, hop 256, 11 groups up to 65 536
    taps) against the reference: complex transform, phase scalogram, offset + time-pooled scalogram."""
    g = load_golden("cqt_high_res.npz")
    cfg = json.loads(str(g["cfg"]))
    x = torch.from_numpy(g["x"]).to(DEV)
    cqt = cpc.CQT(sr=cfg["sample_rate"], fmin=cfg["fmin"], n_bins=cfg["n_bins"], bins_per_octave=cfg["bins_per_octave"],
                  filter_scale=cfg["filter_scale"], hop_length=cfg["hop_length"]).to(DEV)
    assert list(cqt.conv_kernel_sizes) == list(g["kernel_sizes"])
    assert rel_err(cqt(x), g["complex"]) < TOL
    pre = cpc.PreprocessingModule(dict(cfg), phase=True).to(DEV)
    y = pre(x)
    assert tuple(y.shape) == g["phase"].shape
    assert rel_err(y[:, 0], g["phase"][:, 0]) < TOL
    scale = pre.phase_diff.scaling.reshape(-1).cpu()
    assert phase_err_fraction(y[:, 1], g["phase"][:, 1], scale) < 2e-3
    y = cpc.PreprocessingModule(dict(cfg), phase=False, offset_zero=True, pooling=[1, 2]).to(DEV)(x)
    assert rel_err(y, g["offset_pool"]) < TOL


def test_cqt_matches_oracle_on_fresh_input_and_ragged_lengths(cpc):
    plan = O.CqtPlan(16000, 30, 256, 32, 0.5, 128)
    cqt = cpc.CQT(filter_scale=0.5).to(DEV)
    gen = torch.Generator().manual_seed(3)
    for b, extra in [(1, 0), (3, 127), (2, 128 * 3 + 5)]:       # T = 1 (minimum), partial hop, several frames
        x = 0.1 * torch.randn(b, 1, 16384 + 1 + extra, generator=gen)
        want = O.cqt_forward(x, plan)
        got = cqt(x.to(DEV))
        assert tuple(got.shape) == tuple(want.shape)
        assert rel_err(got, want) < TOL
    with pytest.raises(ValueError):
        cqt(torch.zeros(1, 1, 16384, device=DEV))               # one sample short of a frame


def test_cqt_full_size_properties(cpc):
    """BASELINE config-2 size (B=64, L=97024): linearity and hop-shift equivariance."""
    pre = cpc.CQT(filter_scale=0.5).to(DEV)
    gen = torch.Generator(device=DEV).manual_seed(0)
    x = 0.1 * torch.randn(64, 1, 97024, generator=gen, device=DEV)
    z = pre(x)
    assert tuple(z.shape) == (64, 256, 630, 2)
    assert rel_err(pre(2.5 * x), 2.5 * z) < 1e-5
    shifted = pre(x[:, :, 128:].contiguous())
    assert rel_err(shifted, z[:, :, 1:]) < 1e-5


def test_cqt_tensor_core_path_is_fp32_exact(cpc, monkeypatch):
    """The tcgen05 filterbank (fp16 hi/lo planes after exact power-of-two scaling, 22-bit operands) against the oracle's
    filterbank evaluated in float64, next to the errors of the two fp32 evaluations (CUDA-core kernel here, torch CPU
    conv1d in the oracle = what the reference runs): the tensor-core path must be as close to the exact result as an
    fp32 evaluation is.  Inputs cover a loud item, a quiet item (1e-4 of it) and an item with a 100 dB dynamic range."""
    plan = O.CqtPlan(16000, 30, 256, 32, 0.5, 128)
    gen = torch.Generator().manual_seed(5)
    x = 0.1 * torch.randn(3, 1, 16384 + 1 + 128 * 140, generator=gen)
    x[1] *= 1e-4
    x[2, 0, 9000:] *= 1e-5
    exact = O.cqt_forward(x.double(), plan, dtype=torch.float64)
    cpu32 = O.cqt_forward(x, plan)
    cqt = cpc.CQT(filter_scale=0.5).to(DEV)
    res = {}
    for flag in ("0", "1"):
        monkeypatch.setenv("CPC_NO_TENSOR_CQT", flag)
        res[flag] = cqt(x.to(DEV)).cpu()
    errs = {}
    for b in range(3):
        errs[b] = tuple(rel_err(v[b], exact[b]) for v in (res["0"], res["1"], cpu32))
        print("item %d: tensor-core %.2e | CUDA-core fp32 %.2e | torch CPU fp32 %.2e (vs float64)" % ((b,) + errs[b]))
        assert errs[b][0] < 2e-6, errs
        assert errs[b][0] < 4 * max(errs[b][1], errs[b][2]) + 2e-7, errs
    for (lo, hi), k in zip(plan.ranges, plan.kernel_sizes):       # by octave group (diagnostic: error vs filter length)
        print("   K=%5d bins [%3d,%3d): tensor-core %.2e | CUDA-core %.2e | CPU fp32 %.2e" % (
            k, lo, hi, rel_err(res["0"][0, lo:hi], exact[0, lo:hi]), rel_err(res["1"][0, lo:hi], exact[0, lo:hi]),
            rel_err(cpu32[0, lo:hi], exact[0, lo:hi])))
    # the quiet tail of item 2 on its own (frames that only see samples after the drop)
    tail = slice(80, None)
    e_tail = rel_err(res["0"][2, :, tail], exact[2, :, tail])
    print("item 2, quiet tail: tensor-core %.2e" % e_tail)
    assert e_tail < 1e-4


def test_cqt_tensor_core_path_agrees_with_cuda_core_path(cpc):
    """A/B at BASELINE frame counts (T = 630, B = 3): tcgen05 filterbank + fused epilogue against the CUDA-core
    kernels, all three output modes."""
    import os
    gen = torch.Generator().manual_seed(11)
    x = (0.1 * torch.randn(3, 1, 97024, generator=gen)).to(DEV)
    x[1, 0, 30000:60000] = 0.0                                  # a silent stretch: exercises the eps floor / -inf
    d = dict(cpc.cqt_default_dict)
    mods = {"complex": cpc.CQT(filter_scale=0.5).to(DEV),
            "logpow": cpc.PreprocessingModule(d, phase=False, offset_zero=True).to(DEV),
            "phase": cpc.PreprocessingModule(d, phase=True, offset_zero=True, scaling=3.).to(DEV)}
    res = {}
    for flag in ("0", "1"):
        os.environ["CPC_NO_TENSOR_CQT"] = flag
        try:
            res[flag] = {k: m(x).clone() for k, m in mods.items()}
        finally:
            os.environ["CPC_NO_TENSOR_CQT"] = "0"
    assert rel_err(res["0"]["complex"], res["1"]["complex"]) < 5e-5
    assert rel_err(res["0"]["logpow"], res["1"]["logpow"]) < 1e-5
    assert rel_err(res["0"]["phase"][:, 0], res["1"]["phase"][:, 0]) < 1e-5
    scale = 3.0 * mods["phase"].phase_diff.scaling.reshape(-1).cpu()
    loud = res["1"]["logpow"][:, 0, :, 1:] > 0.45               # phase is meaningless where the bin is silent
    a, b = res["0"]["phase"][:, 1], res["1"]["phase"][:, 1]
    dlt = (a - b).cpu().double() / scale.view(1, -1, 1).double()
    dlt = torch.remainder(dlt + math.pi, 2 * math.pi) - math.pi
    assert float((dlt.abs()[loud.cpu()] > 1e-3).double().mean()) < 1e-3


# ---------------------------------------------------------------------------------------------------
# convolution
# ---------------------------------------------------------------------------------------------------

CONV_CASES = [
    # b, cin, h, w, cout, kh, kw, sh, sw, ph, pw, top
    (2, 1, 1, 200, 8, 1, 10, 1, 5, 0, 0, 0),        # AudioEncoder layer 0 shape (C_in = 1)
    (3, 24, 1, 61, 40, 1, 8, 1, 4, 0, 0, 0),        # strided conv1d
    (2, 2, 40, 37, 8, 3, 3, 2, 2, 0, 0, 0),         # first scalogram conv (C_in = 2, stride 2)
    (2, 8, 19, 18, 8, 9, 1, 1, 1, 0, 0, 8),         # tall pitch conv with top-only zero padding
    (2, 8, 19, 18, 16, 3, 3, 2, 2, 1, 1, 0),        # symmetric padding + stride
    (1, 16, 5, 9, 24, 2, 2, 1, 1, 0, 0, 0),
    (2, 70, 3, 7, 130, 1, 1, 1, 1, 2, 2, 0),        # 1x1 residual conv with padding; ragged channel counts
    (1, 3, 6, 6, 5, 6, 6, 1, 1, 0, 0, 0),           # output 1x1
]


@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_forward_backward_match_oracle(cpc, case):
    b, cin, h, w, cout, kh, kw, sh, sw, ph, pw, top = case
    gen = torch.Generator().manual_seed(hash(case) & 0xffff)
    x = torch.randn(b, cin, h, w, generator=gen)
    wt = torch.randn(cout, cin, kh, kw, generator=gen) / math.sqrt(cin * kh * kw)
    bias = torch.randn(cout, generator=gen)
    xr, wr, br = (t.clone().double().requires_grad_(True) for t in (x, wt, bias))
    want = F.conv2d(F.pad(xr, (0, 0, top, 0)), wr, br, stride=(sh, sw), padding=(ph, pw))
    gy = torch.randn(want.shape, generator=gen)
    (want * gy.double()).sum().backward()
    xg, wg, bg = (t.clone().to(DEV).requires_grad_(True) for t in (x, wt, bias))
    got = cpc.ops.conv2d(xg, wg, bg, (sh, sw), (ph, pw), extra_top=top)
    assert tuple(got.shape) == tuple(want.shape)
    assert rel_err(got, want) < TOL
    (got * gy.to(DEV)).sum().backward()
    assert rel_err(xg.grad, xr.grad) < TOL
    assert rel_err(wg.grad, wr.grad) < TOL
    assert rel_err(bg.grad, br.grad) < TOL
    # fused ReLU epilogue + no-bias variant
    got = cpc.ops.conv2d(xg.detach(), wg.detach(), None, (sh, sw), (ph, pw), extra_top=top, relu=True)
    want = F.relu(F.conv2d(F.pad(x.double(), (0, 0, top, 0)), wt.double(), None, stride=(sh, sw), padding=(ph, pw)))
    assert rel_err(got, want) < TOL


UMMA_CASES = [
    # b, cin, h, w, cout, kh, kw, ph, pw, top   (stride 1: the tcgen05 implicit-GEMM path)
    (2, 32, 40, 150, 32, 9, 1, 0, 0, 8),          # tall pitch conv, top-only padding, C_in < 64 (taps share a K chunk)
    (2, 128, 20, 70, 128, 5, 1, 0, 0, 0),         # C_in = 2 K chunks per tap
    (1, 64, 9, 130, 256, 2, 2, 0, 0, 0),          # two N tiles, OW = 129 (three 64-pixel atoms per row)
    (2, 16, 6, 40, 64, 3, 3, 1, 1, 0),            # symmetric padding, 4 taps per K chunk + phantom taps
    (1, 256, 4, 33, 512, 1, 1, 0, 0, 0),          # 1x1, four N tiles
    (3, 32, 1, 300, 96, 1, 5, 0, 0, 0),           # conv1d-shaped (h = 1)
    (2, 64, 3, 8, 128, 1, 1, 2, 2, 0),            # 1x1 residual conv with padding: output wider than input
    (2, 128, 70, 20, 128, 30, 1, 0, 0, 0),        # 30 vertical taps, one channel tile per tap (wgrad M tile = 128 ch)
    (1, 256, 12, 9, 256, 5, 1, 0, 0, 0),          # two channel tiles in wgrad
    # 32 -> 32 channel kh x 1 convs take the row-streaming kernels of conv_tall.cu in fp32 mode
    (1, 32, 50, 200, 32, 64, 1, 0, 0, 63),        # arch-7 block 0 conv_b geometry: most taps of the top rows hit padding
    (3, 32, 37, 64, 32, 16, 1, 0, 0, 0),          # no padding, one atom per row, odd unit count (phantom atom)
    (2, 32, 20, 314, 32, 20, 1, 0, 0, 19),        # kh = tap-ring size, W = 314 (five atoms, last one ragged)
    (1, 32, 8, 40, 32, 8, 1, 0, 0, 3),            # fewer output rows than a tile
    (2, 32, 90, 70, 32, 30, 1, 0, 0, 10),         # several row tiles, partial top padding
    # 128-output-channel kh x 1 convs take conv_tall128.cu (4 output rows per tile, channel-chunk-major)
    (2, 128, 63, 156, 128, 30, 1, 0, 0, 0),       # arch-7 block 1 conv_b geometry
    (1, 128, 9, 64, 128, 4, 1, 0, 0, 3),          # kh = rows per tile, top padding, single atom
    (3, 64, 11, 70, 128, 6, 1, 0, 0, 2),          # one channel chunk forward; dgrad / wgrad fall to the generic kernels
    (1, 256, 13, 40, 128, 7, 1, 0, 0, 0),         # four channel chunks forward
    (2, 128, 12, 30, 64, 5, 1, 0, 0, 4),          # dgrad on the tall kernel (C_in = 128), forward generic
]


@pytest.mark.parametrize("case", UMMA_CASES)
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_tensor_core_conv_matches_oracle(cpc, case, precision):
    b, cin, h, w, cout, kh, kw, ph, pw, top = case
    gen = torch.Generator().manual_seed(hash(case) & 0xffff)
    x = torch.randn(b, cin, h, w, generator=gen)
    wt = torch.randn(cout, cin, kh, kw, generator=gen) / math.sqrt(cin * kh * kw)
    bias = torch.randn(cout, generator=gen)
    xr, wr, br = (t.clone().double().requires_grad_(True) for t in (x, wt, bias))
    want = F.conv2d(F.pad(xr, (0, 0, top, 0)), wr, br, padding=(ph, pw))
    gy = torch.randn(want.shape, generator=gen)
    (want * gy.double()).sum().backward()
    xg, wg, bg = (t.clone().to(DEV).requires_grad_(True) for t in (x, wt, bias))
    got = cpc.ops.conv2d(xg, wg, bg, (1, 1), (ph, pw), extra_top=top, precision=precision)
    assert tuple(got.shape) == tuple(want.shape)
    tol = 5e-5 if precision == "fp32" else 1e-2         # fp32 mode = 3x bf16 split, far inside the 1e-3 budget
    assert rel_err(got, want) < tol
    (got * gy.to(DEV)).sum().backward()
    assert rel_err(xg.grad, xr.grad) < tol
    assert rel_err(wg.grad, wr.grad) < max(tol, TOL)
    assert rel_err(bg.grad, br.grad) < TOL
    got = cpc.ops.conv2d(xg.detach(), wg.detach(), None, (1, 1), (ph, pw), extra_top=top, relu=True, precision=precision)
    want = F.relu(F.conv2d(F.pad(x.double(), (0, 0, top, 0)), wt.double(), None, padding=(ph, pw)))
    assert rel_err(got, want) < tol


@pytest.mark.parametrize("geom", [(32, 127, 314, 64, 63), (128, 63, 156, 30, 0)])
def test_tall_conv_full_size_agrees_with_generic_kernel(cpc, geom):
    """BASELINE-size geometry of the 64x1 and 30x1 pitch convs (B = 4): the row-streaming kernels against the
    generic implicit-GEMM tcgen05 kernels on the same data (size-independent A/B property)."""
    import os
    ch, h, w_, kh, top = geom
    gen = torch.Generator().manual_seed(5)
    x = torch.randn(4, ch, h, w_, generator=gen).to(DEV)
    wt = (torch.randn(ch, ch, kh, 1, generator=gen) / math.sqrt(ch * kh)).to(DEV)
    bias = torch.randn(ch, generator=gen).to(DEV)
    gy = torch.randn(4, ch, h + top - kh + 1, w_, generator=gen).to(DEV)
    outs = []
    for flag in ("0", "1"):
        os.environ["CPC_NO_TALL_CONV"] = flag
        try:
            xg, wg, bg = (t.clone().requires_grad_(True) for t in (x, wt, bias))
            y = cpc.ops.conv2d(xg, wg, bg, (1, 1), (0, 0), extra_top=top)
            (y * gy).sum().backward()
            outs.append((y.detach(), xg.grad, wg.grad, bg.grad))
        finally:
            os.environ["CPC_NO_TALL_CONV"] = "0"
    # y, dx: 5e-5.  dw reduces over 160 k pixels per weight in fp32 accumulators split differently by the two kernels
    # (pixel-chunk shares per CTA), so the two fp32-faithful results differ by a little more: 1e-4, still 10x inside
    # the 1e-3 budget.
    for (a, b), tol in zip(zip(*outs), (5e-5, 5e-5, 1e-4, 1e-4)):
        assert rel_err(a, b) < tol


@pytest.mark.parametrize("geom", [
    # cin, h, w, cout, kh, kw, stride: the arch-7 layers whose rows are not a multiple of 64 pixels wide
    (32, 127, 314, 128, 3, 3, 2),      # block 1 conv_a: output rows of 156 pixels
    (128, 34, 156, 256, 3, 3, 2),      # block 2 conv_a: output rows of 77 pixels
    (256, 16, 77, 256, 15, 1, 1),      # block 2 conv_b: output rows of 77 pixels, 2 rows
])
def test_generic_conv_full_size_matches_torch(cpc, geom):
    """BASELINE-size geometry (B = 2) of the three arch-7 layers on the generic tcgen05 kernels -- rows of 156 / 77
    pixels, i.e. ragged 64-pixel atoms, stride-2 replicas, four dgrad parity classes: forward, data gradient and
    weight gradient against torch's conv2d in float64."""
    cin, h, w_, cout, kh, kw, st = geom
    gen = torch.Generator().manual_seed(6)
    x = torch.randn(2, cin, h, w_, generator=gen)
    wt = torch.randn(cout, cin, kh, kw, generator=gen) / math.sqrt(cin * kh * kw)
    bias = torch.randn(cout, generator=gen)
    xr, wr, br = (t.clone().double().requires_grad_(True) for t in (x, wt, bias))
    want = F.conv2d(xr, wr, br, stride=st)
    gy = torch.randn(want.shape, generator=gen)
    (want * gy.double()).sum().backward()
    xg, wg, bg = (t.clone().to(DEV).requires_grad_(True) for t in (x, wt, bias))
    got = cpc.ops.conv2d(xg, wg, bg, (st, st), (0, 0))
    assert rel_err(got, want) < 5e-5
    (got * gy.to(DEV)).sum().backward()
    assert rel_err(xg.grad, xr.grad) < 5e-5
    assert rel_err(wg.grad, wr.grad) < TOL
    assert rel_err(bg.grad, br.grad) < TOL


UMMA_STRIDED_CASES = [
    # b, cin, h, w, cout, kh, kw, sh, sw, ph, pw, top
    (2, 32, 41, 75, 128, 3, 3, 2, 2, 0, 0, 0),      # arch-7 block 1 conv_a shape (3x3, stride 2)
    (2, 128, 20, 33, 256, 3, 3, 2, 2, 0, 0, 0),     # arch-7 block 2 conv_a shape
    (1, 64, 9, 40, 64, 3, 3, 2, 2, 1, 1, 0),        # stride 2 with symmetric padding
    (2, 64, 1, 203, 64, 1, 8, 1, 4, 0, 0, 0),       # AudioEncoder layer 1 shape (k 8, stride 4)
    (2, 64, 1, 100, 128, 1, 4, 1, 2, 0, 0, 0),      # AudioEncoder layers 2-4 shape (k 4, stride 2)
    (1, 32, 10, 20, 32, 1, 1, 2, 2, 0, 0, 0),       # stride larger than the kernel: some dgrad classes are empty
    (1, 32, 12, 30, 64, 3, 1, 2, 1, 0, 0, 2),       # vertical stride + top padding
    (1, 32, 10, 21, 64, 2, 2, 2, 2, 0, 0, 0),       # class-fused data gradient: every class has exactly one tap
    (2, 32, 11, 20, 64, 4, 4, 2, 2, 0, 0, 0),       # class-fused data gradient: every class has 2 x 2 taps
    (1, 32, 14, 19, 128, 3, 2, 2, 2, 0, 0, 0),      # class-fused, odd width: the last column exists for rw = 0 only
]


@pytest.mark.parametrize("case", UMMA_STRIDED_CASES)
def test_tensor_core_strided_conv_matches_oracle(cpc, case):
    b, cin, h, w, cout, kh, kw, sh, sw, ph, pw, top = case
    gen = torch.Generator().manual_seed(hash(case) & 0xffff)
    x = torch.randn(b, cin, h, w, generator=gen)
    wt = torch.randn(cout, cin, kh, kw, generator=gen) / math.sqrt(cin * kh * kw)
    bias = torch.randn(cout, generator=gen)
    xr, wr, br = (t.clone().double().requires_grad_(True) for t in (x, wt, bias))
    want = F.conv2d(F.pad(xr, (0, 0, top, 0)), wr, br, stride=(sh, sw), padding=(ph, pw))
    gy = torch.randn(want.shape, generator=gen)
    (want * gy.double()).sum().backward()
    xg, wg, bg = (t.clone().to(DEV).requires_grad_(True) for t in (x, wt, bias))
    got = cpc.ops.conv2d(xg, wg, bg, (sh, sw), (ph, pw), extra_top=top)
    assert tuple(got.shape) == tuple(want.shape)
    assert rel_err(got, want) < 5e-5
    (got * gy.to(DEV)).sum().backward()
    assert rel_err(xg.grad, xr.grad) < 5e-5
    assert rel_err(wg.grad, wr.grad) < TOL
    assert rel_err(bg.grad, br.grad) < TOL


def test_audio_encoder_matches_reference_golden(cpc):
    g = load_golden("audio_encoder.npz")
    enc = cpc.AudioEncoder({'strides': [5, 4, 2, 2, 2], 'kernel_sizes': [10, 8, 4, 4, 4],
                            'channel_count': [24, 32, 40, 32, 48], 'bias': True})
    enc.load_state_dict({k[2:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("p.")})
    enc.to(DEV)
    x = torch.from_numpy(g["x"]).to(DEV).requires_grad_(True)
    y = enc(x)
    assert rel_err(y, g["y"]) < TOL
    (y * torch.from_numpy(g["gy"]).to(DEV)).sum().backward()
    assert rel_err(x.grad, g["gx"]) < TOL
    for n, p in enc.named_parameters():
        assert rel_err(p.grad, g["g." + n]) < TOL, n
    # known answers, tests/test_audioEncoder.py:19-48 of the reference
    enc2 = cpc.AudioEncoder({'strides': [5, 4, 2, 2, 2], 'kernel_sizes': [10, 8, 4, 4, 4],
                             'channel_count': [32] * 5, 'bias': True}).to(DEV)
    assert list(enc2(torch.zeros(7, 1, 4800, device=DEV)).shape) == [7, 32, 28]
    with torch.no_grad():
        for p in enc2.parameters():
            p.fill_(0.1)
        imp = torch.zeros(1, 1, 465 + 160, device=DEV)
        base = enc2(imp)[0, 0, 0].item()
        imp[0, 0, 464] = 1.0
        assert enc2(imp)[0, 0, 0].item() != base            # last sample of the receptive field reaches out[0]
        imp.zero_()
        imp[0, 0, 465] = 1.0
        assert enc2(imp)[0, 0, 0].item() == base            # the next one does not


def small_resnet_cfg():
    from test_oracle_golden import small_resnet_blocks
    blocks = small_resnet_blocks()
    blocks[0]['in_channels'] = 1           # the encoder itself sets 2 when phase=True, as in the reference
    return {'phase': True, 'blocks': blocks, 'activation_register': None}


def test_residual_encoder_matches_reference_golden(cpc):
    g = load_golden("resnet_encoder.npz")
    enc = cpc.ScalogramResidualEncoder(small_resnet_cfg())
    sd = {k[2:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("p.")}
    assert set(sd) == set(enc.state_dict()), set(sd) ^ set(enc.state_dict())
    # the golden state holds BN running stats AFTER the forward; reset them to the initial values
    for k in sd:
        if k.endswith("running_mean"):
            sd[k] = torch.zeros_like(sd[k])
        if k.endswith("running_var"):
            sd[k] = torch.ones_like(sd[k])
        if k.endswith("num_batches_tracked"):
            sd[k] = torch.zeros_like(sd[k])
    enc.load_state_dict(sd)
    enc.to(DEV).train()
    x = torch.from_numpy(g["x"]).to(DEV).requires_grad_(True)
    y = enc(x)
    assert tuple(y.shape) == g["y"].shape
    assert rel_err(y, g["y"]) < TOL
    (y * torch.from_numpy(g["gy"]).to(DEV)).sum().backward()
    assert rel_err(x.grad, g["gx"]) < TOL
    noise_only = bn_shadowed_biases(enc.state_dict().keys())
    assert len(noise_only) == 4
    for n, p in enc.named_parameters():
        if n in noise_only:
            assert float(p.grad.abs().max()) < 1e-4, n
            continue
        assert grad_err(p.grad, g["g." + n]) < 2 * TOL, n
    for k, v in enc.state_dict().items():                      # BN running statistics after one step
        if k.endswith("running_mean") or k.endswith("running_var"):
            assert rel_err(v, g["p." + k]) < TOL, k


@pytest.mark.parametrize("tensor_cqt", [False, True])
@pytest.mark.parametrize("tag,phase", [("m", False), ("p", True), ("s", False)])
def test_scalogram_encoder_matches_reference_golden(cpc, monkeypatch, tag, phase, tensor_cqt):
    """ScalogramEncoder (scalogram_model.py:129-227; SURVEY 8a row a6): own CQT -> log power (+ phase difference) ->
    ZeroPad / conv / pool / ReLU / BatchNorm stack, forward and parameter gradients against the reference.  Held to 1e-3
    with the fp32 filterbank; with the tensor-core filterbank the log / atan2 of near-silent cells widens the bound
    (same effect as in the training replays)."""
    monkeypatch.setenv("CPC_NO_TENSOR_CQT", "0" if tensor_cqt else "1")
    full = load_golden("scalogram_encoder.npz")
    g = {k[len(tag) + 1:]: v for k, v in full.items() if k.startswith(tag + ".")}
    cfg = dict(cpc.cqt_default_dict)
    cfg.update({'kernel_sizes': [(9, 1), (5, 5), (5, 1), (3, 3)], 'top_padding': [8, 0, 0, 0],
                'channel_count': [1, 8, 8, 16, 24], 'pooling': [1, 2, 1, 2], 'stride': [1, 1, 1, 1], 'bias': True,
                'batch_norm': True, 'phase': phase, 'separable': tag == "s", 'lowpass_init': 0., 'instance_norm': False,
                'dropout': 0.})                                # tag "s": Conv2dSeparable layers (scalogram_model.py:532-544)
    enc = cpc.ScalogramEncoder(dict(cfg, channel_count=list(cfg['channel_count'])))
    assert enc.receptive_field == int(g["rf"]) and int(enc.downsampling_factor) == int(g["ds"])
    sd = {k[2:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("p.")}
    own = enc.state_dict()
    assert set(sd) == {k for k in own if not k.startswith("cqt.")}, set(sd) ^ {k for k in own if not k.startswith("cqt.")}
    for k in sd:                                                # the golden holds BN statistics AFTER its forward pass
        if k.endswith("running_mean"):
            sd[k] = torch.zeros_like(sd[k])
        if k.endswith("running_var"):
            sd[k] = torch.ones_like(sd[k])
        if k.endswith("num_batches_tracked"):
            sd[k] = torch.zeros_like(sd[k])
    enc.load_state_dict(sd, strict=False)
    enc.to(DEV).train()
    x = torch.from_numpy(g["x"]).to(DEV)
    y = enc(x)
    assert tuple(y.shape) == g["y"].shape
    tol = TOL                                                    # both filterbank paths meet the north-star bound
    assert rel_err(y, g["y"]) < tol
    (y * torch.from_numpy(g["gy"]).to(DEV)).sum().backward()
    for n, p in enc.named_parameters():
        if n.startswith("cqt.") or n.startswith("phase_diff."):
            continue
        # max(tol, 3 x the reference's own gradient noise under a 1e-6 relative change of its CQT output, make_golden.py)
        assert grad_err(p.grad, g["g." + n]) < max(tol, 3.0 * float(g["sn." + n])), (n, float(g["sn." + n]))
    for k in own:
        if k.endswith("running_mean") or k.endswith("running_var"):
            assert rel_err(enc.state_dict()[k], g["p." + k]) < tol, k
    # a trainable filterbank takes the differentiable front end: same values
    if not tensor_cqt and tag != "s":
        enc_t = cpc.ScalogramEncoder(dict(cfg, channel_count=list(cfg['channel_count']), trainable_cqt=True))
        enc_t.load_state_dict(sd, strict=False)
        enc_t.to(DEV).train()
        y_t = enc_t(x)
        assert rel_err(y_t, g["y"]) < tol
        (y_t * torch.from_numpy(g["gy"]).to(DEV)).sum().backward()
        assert all(c.weight.grad is not None and bool(torch.isfinite(c.weight.grad).all()) for c in enc_t.cqt.conv_modules)


# ---------------------------------------------------------------------------------------------------
# max pooling
# ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("shape", [
    dict(b=2, c=8, h=40, w=37, kh=9, kw=1, stride=(1, 1), pad=(0, 0), top=8),
    dict(b=3, c=5, h=21, w=30, kh=5, kw=5, stride=(1, 1), pad=(0, 0), top=0),
    dict(b=2, c=16, h=33, w=41, kh=3, kw=3, stride=(2, 2), pad=(1, 1), top=0),
    dict(b=1, c=32, h=70, w=64, kh=63, kw=1, stride=(1, 1), pad=(0, 0), top=0),
])
def test_depthwise_conv_matches_torch(cpc, shape):
    """cpc_dwconv_* (the depthwise half of Conv2dSeparable) against F.conv2d(groups=C) in float64: forward, data and
    weight gradients."""
    sh = shape
    gen = torch.Generator().manual_seed(13)
    x = torch.randn(sh['b'], sh['c'], sh['h'], sh['w'], generator=gen)
    w = torch.randn(sh['c'], 1, sh['kh'], sh['kw'], generator=gen) / math.sqrt(sh['kh'] * sh['kw'])
    xr, wr = x.double().requires_grad_(True), w.double().requires_grad_(True)
    yr = F.conv2d(F.pad(xr, (0, 0, sh['top'], 0)), wr, None, sh['stride'], sh['pad'], groups=sh['c'])
    gy = torch.randn(yr.shape, generator=gen)
    (yr * gy.double()).sum().backward()
    xg, wg = x.to(DEV).requires_grad_(True), w.to(DEV).requires_grad_(True)
    y = cpc.ops.depthwise_conv2d(xg, wg, sh['stride'], sh['pad'], extra_top=sh['top'])
    assert tuple(y.shape) == tuple(yr.shape)
    (y * gy.to(DEV)).sum().backward()
    assert rel_err(y, yr) < 1e-5 and rel_err(xg.grad, xr.grad) < 1e-5 and rel_err(wg.grad, wr.grad) < 1e-5


@pytest.mark.parametrize("shape,k,ceil", [((2, 3, 9, 11), 2, True), ((2, 3, 9, 11), 2, False), ((1, 5, 12, 12), 3, True),
                                          ((3, 2, 7, 5), 4, True), ((2, 4, 127, 314), 2, True), ((1, 2, 6, 8), 1, False),
                                          ((2, 3, 10, 12), 2, False), ((1, 2, 9, 12), 2, False), ((1, 2, 9, 1030), 2, True)])
def test_max_pool_matches_torch_reference(cpc, shape, k, ceil):
    """nn.MaxPool2d(k, ceil_mode) forward / backward incl. ties (integer-valued input) -- bit exact."""
    gen = torch.Generator().manual_seed(1)
    x = torch.randint(-3, 4, shape, generator=gen).float()          # many ties: first maximum must win
    xr = x.clone().requires_grad_(True)
    yr = F.max_pool2d(xr, k, ceil_mode=ceil)
    gy = torch.randn(yr.shape, generator=gen)
    (yr * gy).sum().backward()
    xg = x.to(DEV).requires_grad_(True)
    yg = cpc.ops.max_pool2d(xg, k, ceil)
    (yg * gy.to(DEV)).sum().backward()
    assert torch.equal(yg.cpu(), yr)
    assert torch.equal(xg.grad.cpu(), xr.grad)


@pytest.mark.parametrize("t,k", [(26, 2), (9, 2), (1, 2), (11, 3)])
def test_ar_max_pool1d_matches_torch(cpc, t, k):
    """ArMaxPool1d (audio_model.py:95-97: MaxPool1d(k, ceil_mode=True)) on the pooling kernels: bit-exact forward and
    backward incl. ties and the ragged last window."""
    from cpc_b200.ar_models import ArMaxPool1d
    gen = torch.Generator().manual_seed(t)
    x = torch.randint(-3, 4, (3, 7, t), generator=gen).float()
    ref = torch.nn.MaxPool1d(k, ceil_mode=True)
    xr = x.clone().requires_grad_(True)
    yr = ref(xr)
    gy = torch.randn(yr.shape, generator=gen)
    (yr * gy).sum().backward()
    xg = x.to(DEV).requires_grad_(True)
    pool = ArMaxPool1d(k, ceil_mode=True)
    assert pool.runs_on_kernels(xg)
    yg = pool(xg)
    (yg * gy.to(DEV)).sum().backward()
    assert torch.equal(yg.cpu(), yr.detach())
    assert torch.equal(xg.grad.cpu(), xr.grad)


@pytest.mark.parametrize("shape,k,ceil", [((2, 4, 21, 38), 2, True), ((2, 3, 20, 37), 2, True), ((1, 5, 19, 31), 3, False)])
def test_conv_and_pool_node_matches_separate_operators(cpc, shape, k, ceil):
    """ops.conv2d_with_pool (one node; the pooling gradient is added in place to the conv's data gradient) against
    conv2d + max_pool2d as two nodes joined by autograd's add: values bit-identical, gradients to fp32 rounding."""
    gen = torch.Generator().manual_seed(21)
    x = torch.randn(shape, generator=gen)
    w = torch.randn(6, shape[1], 3, 3, generator=gen) * 0.2
    b = torch.randn(6, generator=gen)
    outs = []
    for fused in (True, False):
        xg = x.to(DEV).requires_grad_(True)
        wg = w.to(DEV).requires_grad_(True)
        bg = b.to(DEV).requires_grad_(True)
        if fused:
            y, pooled = cpc.ops.conv2d_with_pool(xg, wg, bg, (2, 2), (0, 0), 1, k, ceil)
        else:
            y = cpc.ops.conv2d(xg, wg, bg, (2, 2), (0, 0), 1)
            pooled = cpc.ops.max_pool2d(xg, k, ceil)
        gy = torch.randn(y.shape, generator=torch.Generator().manual_seed(22)).to(DEV)
        gp = torch.randn(pooled.shape, generator=torch.Generator().manual_seed(23)).to(DEV)
        ((y * gy).sum() + (pooled * gp).sum()).backward()
        outs.append((y.detach(), pooled.detach(), xg.grad, wg.grad, bg.grad))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    assert rel_err(outs[0][2], outs[1][2]) < 1e-6
    assert rel_err(outs[0][3], outs[1][3]) < 1e-5 and rel_err(outs[0][4], outs[1][4]) < 1e-5   # split-K atomics: order varies
    # only one branch used downstream
    xg = x.to(DEV).requires_grad_(True)
    y, pooled = cpc.ops.conv2d_with_pool(xg, w.to(DEV), None, (2, 2), (0, 0), 1, k, ceil)
    pooled.sum().backward()
    xr = x.to(DEV).requires_grad_(True)
    cpc.ops.max_pool2d(xr, k, ceil).sum().backward()
    assert torch.equal(xg.grad, xr.grad)


# ---------------------------------------------------------------------------------------------------
# fused BatchNorm + ReLU (+ cropped residual + ReLU)
# ---------------------------------------------------------------------------------------------------

def _bn_reference(x, bn, res, off, relu, outer_relu):
    """CPU restatement of scalogram_model.py:399-431 (bn, relu), :451-472 (crop + add), :523-527 (relu)."""
    y = bn(x)
    if relu:
        y = F.relu(y)
    if res is not None:
        y = y + res[:, :, off[0]:off[0] + y.shape[2], off[1]:off[1] + y.shape[3]]
        if outer_relu:
            y = F.relu(y)
    return y


@pytest.mark.parametrize("shape,res_extra,off,relu,outer,train", [
    ((3, 5, 7, 19), None, (0, 0), True, False, True),
    ((4, 8, 13, 37), (1, 1), (0, 0), True, True, True),
    ((2, 6, 9, 130), (2, 3), (1, 2), True, True, True),
    ((2, 4, 5, 4200), (0, 0), (0, 0), True, False, True),       # more than one segment per plane
    ((3, 7, 6, 11), (1, 0), (1, 0), False, True, True),
    ((2, 5, 8, 33), (1, 1), (0, 1), True, True, False),        # eval(): running statistics
    ((2, 3, 5, 4201), (1, 2), (1, 1), True, True, True),        # saved outer-ReLU bit mask, ragged last mask word
    ((2, 4, 37, 130), (2, 0), (1, 0), False, True, False),      # mask, eval()
])
def test_bn_relu_matches_torch_reference(cpc, shape, res_extra, off, relu, outer, train):
    g = torch.Generator().manual_seed(7)
    b, c, h, w = shape
    x = torch.randn(shape, generator=g) * 2 + 0.5
    res = None if res_extra is None else torch.randn(b, c, h + res_extra[0], w + res_extra[1], generator=g)
    gy = torch.randn(shape, generator=g)

    def make_bn():
        bn = torch.nn.BatchNorm2d(c)
        with torch.no_grad():
            bn.weight.copy_(torch.linspace(0.5, 1.5, c))
            bn.bias.copy_(torch.linspace(-0.3, 0.3, c))
            bn.running_mean.copy_(torch.linspace(-0.2, 0.6, c))
            bn.running_var.copy_(torch.linspace(0.8, 4.0, c))
        return bn.train(train)
    ref_bn, our_bn = make_bn(), make_bn().to(DEV)
    xr = x.clone().requires_grad_(True)
    rr = None if res is None else res.clone().requires_grad_(True)
    yr = _bn_reference(xr, ref_bn, rr, off, relu, outer)
    (yr * gy).sum().backward()
    xo = x.to(DEV).requires_grad_(True)
    ro = None if res is None else res.to(DEV).requires_grad_(True)
    yo = cpc.ops.bn_relu(xo, our_bn, residual=ro, res_off=off, relu=relu, outer_relu=outer)
    (yo * gy.to(DEV)).sum().backward()
    assert rel_err(yo, yr) < 1e-5
    assert rel_err(xo.grad, xr.grad) < 1e-4
    assert rel_err(our_bn.weight.grad, ref_bn.weight.grad) < 1e-4
    assert rel_err(our_bn.bias.grad, ref_bn.bias.grad) < 1e-4
    if res is not None:
        assert rel_err(ro.grad, rr.grad) < 1e-5
    assert rel_err(our_bn.running_mean, ref_bn.running_mean) < 1e-5
    assert rel_err(our_bn.running_var, ref_bn.running_var) < 1e-5
    assert int(our_bn.num_batches_tracked) == int(ref_bn.num_batches_tracked)


def test_bn_saved_relu_mask_equals_recomputed_mask(cpc):
    """The bit mask the forward pass saves for the ReLU behind the residual add gives bit-identical gradients to
    recomputing it from x and the residual (fp32 and packed backward, via the block-tail node)."""
    g = torch.Generator().manual_seed(11)
    x = torch.randn(2, 6, 21, 250, generator=g)
    res = torch.randn(2, 6, 23, 252, generator=g)
    gy = torch.randn(2, 6, 21, 250, generator=g).to(DEV)
    outs = []
    for no_mask in (False, True):
        cpc.ops.kernel_switches["CPC_NO_BN_MASK"] = no_mask
        try:
            bn = torch.nn.BatchNorm2d(6).to(DEV)
            xo = x.to(DEV).requires_grad_(True)
            ro = res.to(DEV).requires_grad_(True)
            yo = cpc.ops.bn_relu(xo, bn, residual=ro, res_off=(1, 2), relu=True, outer_relu=True)
            (yo * gy).sum().backward()
            outs.append((yo.detach(), xo.grad, ro.grad, bn.weight.grad, bn.bias.grad))
        finally:
            cpc.ops.kernel_switches.pop("CPC_NO_BN_MASK", None)
    for a, b in zip(*outs):
        assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------------
# InfoNCE
# ---------------------------------------------------------------------------------------------------

def test_infonce_matches_reference_trainer_golden(cpc):
    g = load_golden("infonce.npz")
    for c in json.loads(str(g["cases"])):
        t = c["tag"]
        pred = torch.from_numpy(g[t + ".pred"]).to(DEV).requires_grad_(True)
        tgt = torch.from_numpy(g[t + ".tgt"]).to(DEV).requires_grad_(True)
        loss, mx, _, _ = cpc.ops.infonce(pred, tgt, c["all_steps"], c["kind"], c["reg"])
        loss.backward()
        assert abs(loss.item() - float(g[t + ".loss"])) < TOL * max(1.0, abs(float(g[t + ".loss"]))), c
        assert abs(mx.item() - float(g[t + ".max"])) < TOL * max(1.0, abs(float(g[t + ".max"]))), c
        assert rel_err(pred.grad, g[t + ".dpred"]) < TOL, c
        assert rel_err(tgt.grad, g[t + ".dtgt"]) < TOL, c


# (150, 3, 96): several tiles per problem on the CUDA-core kernels (E % 64 != 0), per-step regulariser across tiles
@pytest.mark.parametrize("b,k,e", [(64, 16, 512), (8, 12, 512), (33, 5, 100), (70, 1, 64), (150, 3, 96)])
@pytest.mark.parametrize("all_steps", [False, True])
def test_infonce_matches_oracle_native_sizes_and_strided_targets(cpc, b, k, e, all_steps):
    gen = torch.Generator().manual_seed(b * 1000 + k)
    pred = torch.randn(b, k, e, generator=gen) / math.sqrt(e)
    z = torch.randn(b, e, k + 7, generator=gen)                 # targets = strided view z[:, :, -k:] (audio_model.py:197)
    for kind, reg in (("linear", 0.0), ("softplus", 1.0), ("linear", 0.01)):
        want_loss, want_max, want_dp, want_dz = O.infonce_with_grads(pred, z[:, :, -k:], all_steps, kind, reg)
        pg = pred.clone().to(DEV).requires_grad_(True)
        zg = z.clone().to(DEV).requires_grad_(True)
        loss, mx, loss0, mean_s = cpc.ops.infonce(pg, zg[:, :, -k:], all_steps, kind, reg)
        (3.0 * loss).backward()                                  # non-unit upstream gradient
        assert abs(loss.item() - float(want_loss)) < TOL * max(1.0, abs(float(want_loss)))
        assert abs(mx.item() - float(want_max)) < TOL * max(1.0, abs(float(want_max)))
        assert rel_err(pg.grad, 3.0 * want_dp) < TOL
        assert rel_err(zg.grad[:, :, -k:], 3.0 * want_dz) < TOL
        assert float(zg.grad[:, :, :-k].abs().max()) == 0.0
        if reg == 0.0:
            assert abs(loss0.item() - loss.item()) < 1e-6


@pytest.mark.parametrize("b,k,e,all_steps", [(256, 4, 256, False), (200, 3, 128, False), (170, 16, 128, True),
                                             (330, 8, 64, True), (129, 1, 64, False)])
def test_infonce_tensor_core_path_matches_oracle_and_cuda_core_path(cpc, b, k, e, all_steps):
    """tcgen05 InfoNCE (>= 128 candidates, E % 64 == 0) against the fp64 oracle and against the CUDA-core kernels."""
    import os
    gen = torch.Generator().manual_seed(b + 7 * k)
    pred = torch.randn(b, k, e, generator=gen) * (2.0 / math.sqrt(e))
    z = torch.randn(b, e, k + 3, generator=gen)
    for kind in ("linear", "softplus"):
        want_loss, want_max, want_dp, want_dz = O.infonce_with_grads(pred, z[:, :, -k:], all_steps, kind, 0.0)
        res = {}
        for flag in ("0", "1"):
            os.environ["CPC_NO_TENSOR_INFONCE"] = flag
            try:
                pg = pred.clone().to(DEV).requires_grad_(True)
                zg = z.clone().to(DEV).requires_grad_(True)
                loss, mx, _, mean_s = cpc.ops.infonce(pg, zg[:, :, -k:], all_steps, kind, 0.0)
                (2.0 * loss).backward()
                res[flag] = (loss.item(), mx.item(), mean_s.item(), pg.grad.clone(), zg.grad.clone())
            finally:
                os.environ["CPC_NO_TENSOR_INFONCE"] = "0"
        for flag in ("0", "1"):
            loss, mx, mean_s, dp, dz = res[flag]
            assert abs(loss - float(want_loss)) < TOL * max(1.0, abs(float(want_loss))), (flag, kind)
            assert abs(mx - float(want_max)) < TOL * max(1.0, abs(float(want_max))), (flag, kind)
            assert rel_err(dp, 2.0 * want_dp) < TOL, (flag, kind)
            assert rel_err(dz[:, :, -k:], 2.0 * want_dz) < TOL, (flag, kind)
        assert abs(res["0"][2] - res["1"][2]) < 1e-4 * max(1.0, abs(res["1"][2]))
        assert rel_err(res["0"][3], res["1"][3]) < 1e-4 and rel_err(res["0"][4], res["1"][4]) < 1e-4
        # the regulariser (reference default 0.01; exaggerated here) and its gradient on the tensor path: all-steps mode with
        # whole K-groups inside a 128-row tile
        if all_steps and 128 % k == 0:
            want = O.infonce_with_grads(pred, z[:, :, -k:], all_steps, kind, 0.7)
            got = {}
            for flag in ("0", "1"):
                os.environ["CPC_NO_TENSOR_INFONCE"] = flag
                try:
                    pg = pred.clone().to(DEV).requires_grad_(True)
                    zg = z.clone().to(DEV).requires_grad_(True)
                    loss, _, _, _ = cpc.ops.infonce(pg, zg[:, :, -k:], all_steps, kind, 0.7)
                    (2.0 * loss).backward()
                    got[flag] = (loss.item(), pg.grad.clone(), zg.grad[:, :, -k:].clone())
                finally:
                    os.environ["CPC_NO_TENSOR_INFONCE"] = "0"
                assert abs(got[flag][0] - float(want[0])) < TOL * max(1.0, abs(float(want[0]))), (flag, kind)
                assert rel_err(got[flag][1], 2.0 * want[2]) < TOL and rel_err(got[flag][2], 2.0 * want[3]) < TOL, (flag, kind)
            assert rel_err(got["0"][1], got["1"][1]) < 1e-4 and rel_err(got["0"][2], got["1"][2]) < 1e-4
        # bf16 operand mode on the tensor path (one MMA per product instead of three): stated bound 1e-2
        pg = pred.clone().to(DEV).requires_grad_(True)
        zg = z.clone().to(DEV).requires_grad_(True)
        loss, mx, _, _ = cpc.ops.infonce(pg, zg[:, :, -k:], all_steps, kind, 0.0, precision="bf16")
        (2.0 * loss).backward()
        assert abs(loss.item() - float(want_loss)) < 1e-2 * max(1.0, abs(float(want_loss))), kind
        assert rel_err(pg.grad, 2.0 * want_dp) < 1e-2 and rel_err(zg.grad[:, :, -k:], 2.0 * want_dz) < 1e-2, kind


def test_infonce_full_size_property(cpc):
    """Sweep corner the reference cannot materialise (N = 4096 candidates, K = 8): loss of a perfectly
    predictable batch -> ~0 and of an uninformative one -> log N."""
    b, k, e = 4096, 8, 128
    gen = torch.Generator(device=DEV).manual_seed(1)
    z = torch.randn(b, e, k, generator=gen, device=DEV)
    zn = z / z.norm(dim=1, keepdim=True)
    pred = 40.0 * zn.permute(0, 2, 1).contiguous()
    loss, _, _, _ = cpc.ops.infonce(pred, zn, False, "linear", 0.0)
    assert loss.item() < 1e-3
    loss, _, _, _ = cpc.ops.infonce(torch.zeros_like(pred), zn, False, "linear", 0.0)
    assert abs(loss.item() - math.log(b)) < 1e-3


def test_infonce_validate_matches_reference_validate_golden(cpc):
    """cpc_infonce_validate against the reference's own ContrastiveEstimationTrainer.validate() outputs."""
    g = load_golden("validate.npz")
    for c in json.loads(str(g["cases"])):
        t = c["tag"]
        pred = torch.from_numpy(g[t + ".pred"]).to(DEV)
        tgt = torch.from_numpy(g[t + ".tgt"]).to(DEV)
        losses, acc, score = cpc.ops.infonce_validate(pred, tgt, c["all_steps"], c["kind"])
        scale = max(1.0, float(np.abs(g[t + ".losses"]).max()))
        assert float((losses.cpu() - torch.from_numpy(g[t + ".losses"])).abs().max()) < TOL * scale, c
        assert torch.equal(acc.cpu(), torch.from_numpy(g[t + ".acc"])), c          # counts / n: exact
        assert abs(float(score) - float(g[t + ".score"])) < TOL * max(1.0, abs(float(g[t + ".score"]))), c
        want = O.validation_metrics(pred.cpu(), tgt.cpu(), c["all_steps"], c["kind"])
        assert rel_err(losses, want[0]) < TOL and torch.equal(acc.cpu(), want[1])


# ---------------------------------------------------------------------------------------------------
# whole training steps against the reference's own train()
# ---------------------------------------------------------------------------------------------------

def _replay_trainer(cpc, g, model, pre, seed, steps=2, **kw):
    lr, bs = float(g["lr"]), int(g["batch_size"])
    sd0 = {k[3:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("s0.")}
    model.load_state_dict(sd0)
    model.to(DEV)
    if pre is not None:
        pre.to(DEV)
    from cpc_b200.sampler import SyntheticAudioDataset

    class Items(torch.utils.data.Dataset):
        def __init__(self, items):
            self.items = items

        def __len__(self):
            return self.items.shape[0]

        def __getitem__(self, i):
            return self.items[i]

        def get_example_count_per_file(self):
            return [len(self)]

    class Log:
        def __init__(self):
            self.l, self.s = [], []
            outer = self

            class M:
                def __init__(self, sink):
                    self.sink = sink

                def update(self, v, n=1):
                    self.sink.append(v)

            self.loss_meter, self.score_meter = M(self.l), M(self.s)

        def log(self, step):
            pass

    log = Log()
    trainer = cpc.ContrastiveEstimationTrainer(model=model, dataset=Items(torch.from_numpy(g["items"])), logger=log,
                                               device=DEV, optimizer=torch.optim.SGD, preprocessing=pre,
                                               verbose=False, **kw)
    random.seed(seed)
    snaps = []
    for s in range(steps):
        trainer.train(batch_size=bs, epochs=1, lr=lr, continue_training_at_step=s, num_workers=0, max_steps=s + 1)
        snaps.append({k: v.detach().cpu().clone() for k, v in model.state_dict().items()})
    return log, snaps, lr


def _check_against_snapshots(g, log, snaps, lr, tol, drift_tol=None):
    worst = {"loss": 0.0, "grad": 0.0, "param": 0.0, "drift": 0.0}
    drift_tol = tol if drift_tol is None else drift_tol
    for s in range(len(snaps)):
        worst["loss"] = max(worst["loss"], abs(log.l[s] - g["losses"][s]) / max(1.0, abs(g["losses"][s])))
        assert abs(log.l[s] - g["losses"][s]) < tol * max(1.0, abs(g["losses"][s])), (s, log.l, g["losses"])
        assert abs(log.s[s] - g["max_scores"][s]) < tol * max(1.0, abs(g["max_scores"][s]))
    # step-1 gradients: (before - after) / lr for every float parameter, reference vs ours
    noise_only = bn_shadowed_biases(snaps[0].keys())
    for k, after in snaps[0].items():
        if not after.dtype.is_floating_point or k.endswith("running_mean") or k.endswith("running_var"):
            continue
        if k in noise_only:
            continue
        before = torch.from_numpy(g["s0." + k])
        ref_grad = (before - torch.from_numpy(g["s1." + k])) / lr
        my_grad = (before - after) / lr
        worst["grad"] = max(worst["grad"], grad_err(my_grad, ref_grad))
        assert grad_err(my_grad, ref_grad) < tol, k
    for k, after in snaps[-1].items():
        if not after.dtype.is_floating_point:
            continue
        want = torch.from_numpy(g["s%d.%s" % (len(snaps), k)])
        if k in noise_only:
            # a conv bias in front of a batch norm has an exactly-zero true gradient: both sides integrate
            # rounding noise, so only closeness in absolute terms is meaningful
            assert float((after - want).abs().max()) < 1e-4, k
            continue
        if float(torch.from_numpy(g["s0." + k]).abs().max()) == 0.0:
            # zero-initialised parameters (batch-norm shifts): the value IS the accumulated update, i.e. a sum of
            # per-step gradients along the two trajectories, relative to a quantity that starts at zero
            worst["drift"] = max(worst["drift"], rel_err(after, want))
            assert rel_err(after, want) < drift_tol, k
            continue
        worst["param"] = max(worst["param"], rel_err(after, want))
        assert rel_err(after, want) < tol, k
    print("replay vs reference train(): worst relative errors %s (bounds %g, drift %g)"
          % ({k: float("%.2g" % v) for k, v in worst.items()}, tol, drift_tol))


def test_training_steps_raw_wave_match_reference_train(cpc):
    g = load_golden("trainer_raw.npz")
    enc = cpc.AudioEncoder({'strides': [5, 4, 2, 2, 2], 'kernel_sizes': [10, 8, 4, 4, 4],
                            'channel_count': [16, 24, 24, 24, 32], 'bias': True})
    model = cpc.AudioPredictiveCodingModel(enc, cpc.AudioGRUModel(32, 16), enc_size=32, ar_size=16, visible_steps=9,
                                           prediction_steps=4)
    log, snaps, lr = _replay_trainer(cpc, g, model, None, seed=0, regularization=1., score_over_all_timesteps=False,
                                     score_function=cpc.softplus_score_function, prediction_steps=4)
    _check_against_snapshots(g, log, snaps, lr, TOL)


def test_training_steps_cqt_resnet_match_reference_train(cpc):
    g = load_golden("trainer_cqt.npz")
    cfg = small_resnet_cfg()
    cfg['blocks'][2] = dict(cfg['blocks'][2], kernel_size_1=(30, 2), pooling_1=1, ceil_pooling=False)
    cfg['blocks'][1] = dict(cfg['blocks'][1], kernel_size_2=(35, 1))
    pre = cpc.PreprocessingModule(dict(cpc.cqt_default_dict), phase=True)
    enc = cpc.ScalogramResidualEncoder(cfg, preprocessing_module=pre)
    ar = cpc.ConvolutionalArModel({'kernel_sizes': [3, 3], 'channel_count': [24, 16, 16], 'stride': [1, 1],
                                   'pooling': [1, 2], 'bias': True, 'batch_norm': True, 'residual': False,
                                   'activation_register': None})
    model = cpc.AudioPredictiveCodingModel(enc, ar, enc_size=24, ar_size=16, visible_steps=10, prediction_steps=3)
    assert model.item_length == int(g["item_length"])
    log, snaps, lr = _replay_trainer(cpc, g, model, pre, seed=3, steps=3, regularization=0.25, score_over_all_timesteps=True,
                                     score_function=cpc.linear_score_function, prediction_steps=3)
    _check_against_snapshots(g, log, snaps, lr, TOL)


@pytest.mark.parametrize("tensor_cqt", [False, True])
@pytest.mark.parametrize("tag,all_steps", [("a", True), ("p", False)])
def test_training_steps_gradient_penalty_match_reference_train(cpc, monkeypatch, tag, all_steps, tensor_cqt):
    """wasserstein_gradient_penalty=True (contrastive_estimation_training.py:144-158): two SGD steps of the reference
    trainer, replayed.  The penalty needs d/dparams of ||d sum(scores) / d scalogram||, i.e. the second derivative
    of every encoder conv (dgrad / wgrad / forward kernels chained through autograd) and of the AR model.

    Both filterbanks (fp32 CUDA-core kernel and the default fp16 hi/lo tensor-core kernel) are held to 1e-3; measured
    worst gradient error 2e-4 (round 1's bf16 hi/lo filterbank, 1e-5 relative, needed 5e-2 here: the penalty differentiates
    the log / atan2 of near-silent CQT cells, tools/diag_training_gp.py)."""
    monkeypatch.setenv("CPC_NO_TENSOR_CQT", "0" if tensor_cqt else "1")
    full = load_golden("trainer_gp.npz")
    g = {k[len(tag) + 1:]: v for k, v in full.items() if k.startswith(tag + ".")}
    cfg = small_resnet_cfg()
    cfg['blocks'][2] = dict(cfg['blocks'][2], kernel_size_1=(30, 2), pooling_1=1, ceil_pooling=False)
    cfg['blocks'][1] = dict(cfg['blocks'][1], kernel_size_2=(35, 1))
    pre = cpc.PreprocessingModule(dict(cpc.cqt_default_dict), phase=True)
    enc = cpc.ScalogramResidualEncoder(cfg, preprocessing_module=pre)
    ar = cpc.ConvolutionalArModel({'kernel_sizes': [3, 3], 'channel_count': [24, 16, 16], 'stride': [1, 1],
                                   'pooling': [1, 2], 'bias': True, 'batch_norm': True, 'residual': False,
                                   'activation_register': None})
    model = cpc.AudioPredictiveCodingModel(enc, ar, enc_size=24, ar_size=16, visible_steps=10, prediction_steps=3)
    assert model.item_length == int(g["item_length"])
    fn = cpc.linear_score_function if all_steps else cpc.softplus_score_function
    log, snaps, lr = _replay_trainer(cpc, g, model, pre, seed=5, steps=2, regularization=0.25,
                                     score_over_all_timesteps=all_steps, score_function=fn, prediction_steps=3,
                                     wasserstein_gradient_penalty=True, gradient_penalty_factor=10.)
    _check_against_snapshots(g, log, snaps, lr, TOL)


@pytest.mark.parametrize("shape", [
    dict(b=3, ci=5, co=6, h=11, w=13, kh=3, kw=3, stride=(2, 2), pad=(1, 1), top=0),       # cuda-core family
    dict(b=2, ci=32, co=32, h=40, w=70, kh=9, kw=1, stride=(1, 1), pad=(0, 0), top=8),     # tall 32-channel family
    dict(b=2, ci=32, co=64, h=21, w=72, kh=3, kw=3, stride=(2, 2), pad=(0, 0), top=0),     # generic tcgen05 family
    dict(b=2, ci=2, co=32, h=30, w=41, kh=3, kw=3, stride=(2, 2), pad=(0, 0), top=0),      # small-K family
])
def test_conv_second_derivatives_match_torch(cpc, shape):
    """Backward-of-backward of the conv Function: L = sum((d<y, gy>/dx)^2) + sum((d<y, gy>/dw)^2) differentiated
    w.r.t. x, w and gy, against the same expression built from torch's conv2d in float64 on the CPU."""
    gen = torch.Generator().manual_seed(21)
    sh = shape
    x = torch.randn(sh['b'], sh['ci'], sh['h'], sh['w'], generator=gen)
    w = torch.randn(sh['co'], sh['ci'], sh['kh'], sh['kw'], generator=gen) / math.sqrt(sh['ci'] * sh['kh'] * sh['kw'])
    bias = torch.randn(sh['co'], generator=gen)

    def second(conv, x, w, bias, gy=None):
        x, w, bias = x.requires_grad_(True), w.requires_grad_(True), bias.requires_grad_(True)
        y = conv(x, w, bias)
        if gy is None:
            gy = torch.randn(y.shape, generator=torch.Generator().manual_seed(22))
        gy = gy.to(device=y.device, dtype=y.dtype).requires_grad_(True)
        gx, gw = torch.autograd.grad((y * gy).sum(), (x, w), create_graph=True)
        loss = (gx ** 2).sum() + (gw ** 2).sum()
        return [gx, gw] + list(torch.autograd.grad(loss, (x, w, gy)))

    mine = second(lambda x, w, b: cpc.ops.conv2d(x, w, b, sh['stride'], sh['pad'], extra_top=sh['top']),
                  x.clone().to(DEV), w.clone().to(DEV), bias.clone().to(DEV))
    ref = second(lambda x, w, b: F.conv2d(F.pad(x, (0, 0, sh['top'], 0)), w, b, sh['stride'], sh['pad']),
                 x.double(), w.double(), bias.double())
    for name, a, b in zip(("gx", "gw", "dL/dx", "dL/dw", "dL/dgy"), mine, ref):
        assert rel_err(a, b) < TOL, name


def test_fused_functions_refuse_second_derivatives(cpc):
    """The fused BN+ReLU / pooling / InfoNCE backward kernels are first-order only: asking autograd to differentiate
    them again must raise instead of silently returning a constant."""
    x = torch.randn(2, 4, 6, 8, device=DEV, requires_grad=True)
    y = cpc.ops.max_pool2d(x, 2)
    (gx,) = torch.autograd.grad(y.sum(), x, create_graph=True)
    with pytest.raises(RuntimeError):
        torch.autograd.grad((gx ** 2).sum(), x)


@pytest.mark.parametrize("fused_adam", [False, True])
def test_cuda_graph_step_reproduces_eager_steps(cpc, fused_adam):
    """GraphedTrainStep (one captured CUDA graph per step) against the same steps submitted eagerly with
    torch.optim.Adam; with the stock optimizer and with the single-kernel cpc_b200.optim.Adam inside the graph."""
    def make(fused=False):
        torch.manual_seed(5)
        cfg = small_resnet_cfg()
        cfg['blocks'][2] = dict(cfg['blocks'][2], kernel_size_1=(30, 2), pooling_1=1, ceil_pooling=False)
        cfg['blocks'][1] = dict(cfg['blocks'][1], kernel_size_2=(35, 1))
        pre = cpc.PreprocessingModule(dict(cpc.cqt_default_dict), phase=True)
        enc = cpc.ScalogramResidualEncoder(cfg, preprocessing_module=pre)
        ar = cpc.ConvolutionalArModel({'kernel_sizes': [3, 3], 'channel_count': [24, 16, 16], 'stride': [1, 1],
                                       'pooling': [1, 2], 'bias': True, 'batch_norm': True, 'residual': False,
                                       'activation_register': None})
        model = cpc.AudioPredictiveCodingModel(enc, ar, enc_size=24, ar_size=16, visible_steps=10, prediction_steps=3)
        model.to(DEV).train()
        pre.to(DEV)
        trainer = cpc.ContrastiveEstimationTrainer(model=model, dataset=None, device=torch.device(DEV), regularization=0.1,
                                                   score_over_all_timesteps=True,
                                                   score_function=cpc.linear_score_function, preprocessing=pre,
                                                   prediction_steps=3, verbose=False)
        if fused:
            opt = trainer.make_optimizer(1e-3)
            assert isinstance(opt, cpc.optim.Adam)
        else:
            opt = torch.optim.Adam(model.parameters(), lr=1e-3, capturable=True)
        return model, trainer, opt
    gen = torch.Generator().manual_seed(9)
    model, trainer, opt = make()
    batches = [0.1 * torch.randn(4, model.item_length, generator=gen) for _ in range(3)]
    eager = []
    for x in batches:
        loss, _ = trainer.loss_on_batch(x.to(DEV))
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        eager.append(loss.item())
    model2, trainer2, opt2 = make(fused_adam)
    step = cpc.GraphedTrainStep(trainer2, opt2, (4, model2.item_length), warmup=2)
    graphed = [step(x.pin_memory())[0].item() for x in batches]
    for a, b in zip(eager, graphed):
        assert abs(a - b) < 1e-4 * max(1.0, abs(a)), (eager, graphed)
    # conv biases in front of a batch norm have zero true gradient: Adam turns their rounding noise (atomics order)
    # into lr-sized steps, so they are not comparable between two runs of ANY implementation
    noise_only = bn_shadowed_biases(model.state_dict().keys())
    # ... and an entry whose gradient passes through zero during these steps takes Adam updates that differ by a few
    # percent of lr between two runs: parameters are compared with that absolute slack (2 % of three lr-sized steps)
    for (n, p), (_, q) in zip(model.named_parameters(), model2.named_parameters()):
        if n not in noise_only:
            slack = 1e-4 * float(p.detach().abs().max()) + 0.02 * 3 * 1e-3
            assert float((q.detach() - p.detach()).abs().max()) < slack, (n, float((q.detach() - p.detach()).abs().max()), slack)


@pytest.mark.parametrize("name", ["e24", "e25", "e20"])
def test_experiment_configs_train_one_step(cpc, name):
    """The reference's experiment dicts (conv AR, per-step scoring, attention AR) drive the B200 path unchanged:
    setup_model -> trainer -> one optimisation step at the full item length, small batch."""
    exp = cpc.configs.experiment(name)
    tc = exp["training_config"]
    torch.manual_seed(0)
    model, pre, _ = cpc.configs.setup_model(exp["cqt_config"], exp["encoder_config"], exp["ar_model_config"], tc,
                                            device=torch.device(DEV))
    assert model.item_length == 97024
    trainer = cpc.ContrastiveEstimationTrainer(model=model, dataset=None, device=torch.device(DEV),
                                               regularization=tc["regularization"],
                                               score_over_all_timesteps=tc["score_over_all_timesteps"],
                                               score_function=tc["score_function"], preprocessing=pre,
                                               prediction_steps=tc["prediction_steps"], verbose=False)
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)
    model.train()
    x = 0.1 * torch.randn(8, model.item_length, generator=torch.Generator().manual_seed(2))
    losses = []
    for _ in range(2):
        loss, max_score = trainer.loss_on_batch(x.to(DEV))
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert all(math.isfinite(v) for v in losses), losses
    n = 8 * tc["prediction_steps"] if tc["score_over_all_timesteps"] else 8
    assert losses[0] < 3.0 * math.log(n) + 60.0             # untrained model: within sight of the uniform-softmax loss
    assert all(p.grad is not None and bool(torch.isfinite(p.grad).all()) for p in model.parameters())


def test_gru_model_cudnn_sequence_call_matches_the_cell_loop(cpc):
    """AudioGRUModel on the device: one fused cuDNN GRU call over the 100 visible steps (BASELINE configs[0] geometry:
    512 -> 256) against the unrolled GRUCell loop in float64 -- hidden state and every gradient at fp32 rounding."""
    import copy
    torch.manual_seed(3)
    fused = cpc.AudioGRUModel(512, 256).to(DEV)
    loop = copy.deepcopy(fused).double()
    loop.fused = False
    x = torch.randn(8, 512, 100, generator=torch.Generator().manual_seed(4))
    xa, xb = x.clone().to(DEV).requires_grad_(True), x.clone().to(DEV).double().requires_grad_(True)
    assert fused._use_fused(xa) and not loop._use_fused(xb)
    ya, yb = fused(xa), loop(xb)
    assert rel_err(ya, yb) < 1e-5
    g = torch.randn(ya.shape, generator=torch.Generator().manual_seed(5)).to(DEV)
    (ya * g).sum().backward()
    (yb * g.double()).sum().backward()
    assert rel_err(xa.grad, xb.grad) < 1e-4
    for (n, p_), (_, q_) in zip(fused.named_parameters(), loop.named_parameters()):
        assert rel_err(p_.grad, q_.grad) < 1e-4, n
    with cpc.ops.second_order():                                     # the gradient penalty needs a twice-differentiable path
        assert not fused._use_fused(xa)


def test_bf16_mode_tracks_fp32_mode_on_e20(cpc):
    """BASELINE configs[2] (arch 7 + attention AR in the bf16 operand mode: row-streaming and generic conv kernels on the
    hi plane only, block-tail nodes handing over one plane, the filterbank on one fp16 plane per operand, AR model and W_k
    under bf16 autocast) against the fp32-faithful
    mode of the same model on the same batch.  Per-op error of the mode is <= 1e-2 (conv tests above); through the whole
    network the encoder output is held to 3e-2 and the loss to 2e-2 relative."""
    exp = cpc.configs.experiment("e20")
    tc = exp["training_config"]
    torch.manual_seed(0)
    dev = torch.device(DEV)
    model, pre, _ = cpc.configs.setup_model(exp["cqt_config"], exp["encoder_config"], exp["ar_model_config"], tc, device=dev)
    trainer = cpc.ContrastiveEstimationTrainer(model=model, dataset=None, device=dev, regularization=tc["regularization"],
                                               score_over_all_timesteps=tc["score_over_all_timesteps"],
                                               score_function=tc["score_function"], preprocessing=pre,
                                               prediction_steps=tc["prediction_steps"], verbose=False)
    model.train()
    for m in model.modules():
        if isinstance(m, torch.nn.Dropout):
            m.p = 0.0                                            # the two passes must see the same network
    x = (0.1 * torch.randn(4, model.item_length, generator=torch.Generator().manual_seed(3))).to(DEV)
    results = {}
    for precision in ("fp32", "bf16"):
        cpc.ops.set_default_precision(precision)
        try:
            scal = pre(x.unsqueeze(1))
            code = model.encoder(scal)
            loss, max_score = trainer.loss_on_batch(x)
            model.zero_grad(set_to_none=True)
            loss.backward()
            grads = {n: p.grad.clone() for n, p in model.named_parameters()}
            results[precision] = (code.detach(), float(loss), float(max_score), grads, scal.detach().clone())
        finally:
            cpc.ops.set_default_precision("fp32")
    (c32, l32, m32, g32, s32), (c16, l16, m16, g16, s16) = results["fp32"], results["bf16"]
    print("e20 fp32 / bf16 mode: loss %.6f / %.6f, max score %.5f / %.5f, encoder output rel err %.2e, scalogram rel err "
          "%.2e (log-power) %.2e (phase)" % (l32, l16, m32, m16, rel_err(c16, c32), rel_err(s16[:, 0], s32[:, 0]),
                                             rel_err(s16[:, 1], s32[:, 1])))
    # front end of the mode: one fp16 plane per operand (CPC_CQT_FLAG_HALF_OPERANDS), ~2e-4 per filter response
    # (log-power 1.5e-4 norm-wise; the phase-difference channel is compared on the circle: a bin within rounding of +-pi
    # unwraps the other way, which is 2.9e-2 norm-wise but the same angle)
    assert rel_err(s16[:, 0], s32[:, 0]) < 1e-3
    assert phase_err_fraction(s16[:, 1], s32[:, 1], pre.phase_diff.scaling.reshape(-1).cpu(), tol=2e-2) < 1e-2
    assert rel_err(c16, c32) < 3e-2
    assert abs(l16 - l32) < 2e-2 * abs(l32)
    assert all(bool(torch.isfinite(g).all()) for g in g16.values())
    # same descent direction (ReLU / max-pool gates flip on individual entries under 4e-3 operand rounding, so the
    # gradients are compared by angle over all parameters, not entry by entry)
    flat32 = torch.cat([g32[n].flatten().double() for n in g32])
    flat16 = torch.cat([g16[n].flatten().double() for n in g32])
    cos = float(torch.dot(flat32, flat16) / (flat32.norm() * flat16.norm()))
    print("cosine of the bf16-mode and fp32-mode gradients: %.4f" % cos)
    assert cos > 0.7


@pytest.mark.parametrize("name", ["e29", "e32"])
def test_high_res_experiments_train_one_step(cpc, name):
    """The reference's DEFAULT experiment (e29, train_script.py:11) and the last one (e32), built from the reference's own
    experiment dicts as imported (tests/golden/configs.json): 44.1 kHz / 292-bin / hop-256 filterbank (11 octave groups up
    to 65 536 taps), offset + pooled scalogram, resnet arch 9, attention AR, Wasserstein gradient penalty (second-order
    autograd through the conv kernels).  One optimisation step at the full item length, batch 2."""
    plain = load_golden("configs.json")[name]
    exp = cpc.configs.experiment_from_plain(plain)
    tc = exp["training_config"]
    torch.manual_seed(0)
    dev = torch.device(DEV)
    model, pre, _ = cpc.configs.setup_model(exp["cqt_config"], exp["encoder_config"], exp["ar_model_config"], tc, device=dev)
    want = load_golden("configs_all.json")[name]
    assert model.item_length == want["item_length"]
    assert {n: list(p.shape) for n, p in model.named_parameters()} == want["params"]
    trainer = cpc.ContrastiveEstimationTrainer(model=model, dataset=None, device=dev, regularization=tc["regularization"],
                                               score_over_all_timesteps=tc["score_over_all_timesteps"],
                                               score_function=tc["score_function"], preprocessing=pre,
                                               prediction_steps=tc["prediction_steps"],
                                               wasserstein_gradient_penalty=tc["wasserstein_gradient_penalty"],
                                               gradient_penalty_factor=tc["gradient_penalty_factor"], verbose=False)
    opt = trainer.make_optimizer(tc["learning_rate"])
    model.train()
    x = 0.1 * torch.randn(2, model.item_length, generator=torch.Generator().manual_seed(3))
    losses = []
    for _ in range(2):
        loss, max_score = trainer.loss_on_batch(x.to(DEV))
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert all(math.isfinite(v) for v in losses), losses
    assert all(p.grad is not None and bool(torch.isfinite(p.grad).all()) for p in model.parameters())
    print(name, "item length", model.item_length, "losses", losses, "gradient penalty", tc["wasserstein_gradient_penalty"])


def test_e29_default_experiment_step_matches_reference_golden(cpc):
    """The reference's default experiment e29 at the full item length (367 616 samples, batch 2): the loss the reference's
    own setup_model + train() logs for its first step (InfoNCE + Wasserstein gradient penalty), its max score and the
    encoder output (tests/golden/e29_step.npz, oracle/make_golden.py::golden_e29; attention dropout 0, seeded weights).
    Covers the hop-256 filterbank (CUDA-core kernels + pooled scalogram), resnet arch 9 and the second-order path at size.
    The penalty is a function of d(scores)/d(scalogram), i.e. of the ReLU gate pattern: its tolerance is the gate-noise
    level discussed in DESIGN.md section 2, the forward quantities keep 1e-3."""
    import cpc_oracle_model as OM
    g = load_golden("e29_step.npz")
    plain = load_golden("configs.json")["e29"]
    plain["ar_model_config"]["dropout"] = 0.0
    exp = cpc.configs.experiment_from_plain(plain)
    tc = exp["training_config"]
    torch.manual_seed(0)
    dev = torch.device(DEV)
    model, pre, _ = cpc.configs.setup_model(exp["cqt_config"], exp["encoder_config"], exp["ar_model_config"], tc, device=dev)
    assert model.item_length == int(g["item_length"])
    assert [n for n, _ in model.named_parameters()] == json.loads(str(g["names"]))
    OM.reseed_parameters(model.named_parameters())
    trainer = cpc.ContrastiveEstimationTrainer(model=model, dataset=None, device=dev, regularization=tc["regularization"],
                                               score_over_all_timesteps=tc["score_over_all_timesteps"],
                                               score_function=tc["score_function"], preprocessing=pre,
                                               prediction_steps=tc["prediction_steps"],
                                               wasserstein_gradient_penalty=tc["wasserstein_gradient_penalty"],
                                               gradient_penalty_factor=tc["gradient_penalty_factor"], verbose=False)
    batch, order = int(g["batch"]), [int(i) for i in g["order"]]
    audio = OM.e24_audio(2 * batch, model.item_length, seed=1234)
    assert np.array_equal(audio[:, ::4099].numpy(), g["audio_check"])
    model.train()
    seen = {}
    hook = model.encoder.register_forward_hook(lambda m, i, o: seen.__setitem__("z", o.detach().clone()))
    loss, mx = trainer.loss_on_batch(audio[order[:batch]].to(dev))
    hook.remove()
    loss.backward()
    print("e29 golden: loss %.6f vs %.6f, max score %.6f vs %.6f, z err %.2e" % (
        loss.item(), float(g["losses"][0]), mx.item(), float(g["max_scores"][0]), rel_err(seen["z"], g["z"])))
    assert rel_err(seen["z"], g["z"]) < TOL
    assert abs(mx.item() - float(g["max_scores"][0])) < TOL * abs(float(g["max_scores"][0]))
    # the reference's own loss moves by loss_snl (0.35 %) / loss_snl5 (1.7 %) when each of its conv outputs moves by 2e-6 / 5e-6
    # relative (its encoder output then moves by 7e-5 / 1.8e-4; the CUDA path's differs by 1.2e-4): bound = 3 x the larger
    bound = max(TOL, 3.0 * max(float(g["loss_snl"]), float(g["loss_snl5"])))
    assert abs(loss.item() - float(g["losses"][0])) < bound * abs(float(g["losses"][0])), (loss.item(), float(g["losses"][0]), bound)
    assert all(p.grad is not None and bool(torch.isfinite(p.grad).all()) for p in model.parameters())


@pytest.mark.parametrize("graphed", [False, True])
def test_e24_full_size_training_steps_match_reference_golden(cpc, graphed):
    """BASELINE configs[1] itself, at the full item length, on the path bench.py measures (tensor-core CQT, block-tail
    nodes, single-kernel Adam, optionally the whole step as one CUDA graph): two training steps of
    setup_model(experiments['e24']) against the reference's own setup_model + train() (tests/golden/e24_step.npz,
    oracle/make_golden.py::golden_e24).  Scalogram, encoder output, loss and max score are held to 1e-3; gradients to
    max(1e-3, 3 x the self-noise the reference shows under a 1-ulp-sized change of its scalogram) -- see
    tests/test_oracle_golden.py::check_e24_against_golden."""
    import cpc_oracle_model as OM
    from test_oracle_golden import check_e24_against_golden
    g = load_golden("e24_step.npz")
    names = json.loads(str(g["names"]))
    exp = cpc.configs.experiment("e24")
    tc = exp["training_config"]
    torch.manual_seed(0)
    dev = torch.device(DEV)
    model, pre, _ = cpc.configs.setup_model(exp["cqt_config"], exp["encoder_config"], exp["ar_model_config"], tc, device=dev)
    assert model.item_length == int(g["item_length"])
    assert [n for n, _ in model.named_parameters()] == names         # same state_dict keys, same order as the reference
    OM.reseed_parameters(model.named_parameters())
    assert tc["score_function"] is cpc.linear_score_function and str(g["score_kind"]) == "linear_score_function"
    assert bool(tc["score_over_all_timesteps"]) == bool(g["all_steps"]) and tc["regularization"] == float(g["regularization"])
    trainer = cpc.ContrastiveEstimationTrainer(model=model, dataset=None, device=dev, regularization=tc["regularization"],
                                               score_over_all_timesteps=tc["score_over_all_timesteps"],
                                               score_function=tc["score_function"], preprocessing=pre,
                                               prediction_steps=tc["prediction_steps"], verbose=False)
    batch, order = int(g["batch"]), [int(i) for i in g["order"]]
    audio = OM.e24_audio(2 * batch, model.item_length, seed=int(g["audio_seed"]))
    assert np.array_equal(audio[:, ::4099].numpy(), g["audio_check"])
    batches = [audio[order[i * batch:(i + 1) * batch]] for i in range(2)]
    # the scalogram the encoder sees
    scal = pre(batches[0].to(dev).unsqueeze(1))
    assert tuple(scal.shape) == tuple(int(v) for v in g["scal_shape"])
    assert rel_err(scal[:, 0, ::7, ::11], g["scal_power_sub"]) < TOL
    scale = pre.phase_diff.scaling.reshape(-1).cpu()[::7]
    assert phase_err_fraction(scal[:, 1, ::7, ::11], g["scal_phase_sub"], scale) < 2e-3
    model.train()
    opt = trainer.make_optimizer(float(g["lr"]))
    assert isinstance(opt, cpc.optim.Adam)
    seen = {}
    hook = model.encoder.register_forward_hook(lambda m, i, o: seen.__setitem__("z", o.detach()))
    losses, maxes = [], []
    if graphed:
        step = cpc.GraphedTrainStep(trainer, opt, (batch, model.item_length), warmup=2)
        for i, x in enumerate(batches):
            loss, mx = step(x.pin_memory())
            torch.cuda.synchronize()
            losses.append(loss.item())
            maxes.append(mx.item())
            if i == 0:
                grads = {n: p.grad.detach().clone() for n, p in model.named_parameters()}
                z1 = seen["z"].clone()                          # the graph's static encoder output, rewritten every replay
    else:
        for i, x in enumerate(batches):
            loss, mx = trainer.loss_on_batch(x.to(dev))
            opt.zero_grad(set_to_none=True)
            loss.backward()
            if i == 0:
                grads = {n: p.grad.detach().clone() for n, p in model.named_parameters()}
                z1 = seen["z"].clone()
            opt.step()
            losses.append(loss.item())
            maxes.append(mx.item())
    hook.remove()
    report = check_e24_against_golden(g, names, losses, maxes, z1, grads, dict(model.named_parameters()), tol=TOL,
                                      update_tol=2e-2)
    worst = sorted(((v[0], v[1], k) for k, v in report.items() if not k.startswith("__")), reverse=True)[:3]
    print("e24 golden (graphed=%s): losses %s vs %s; worst gradient errors %s; update mismatch %.4f"
          % (graphed, losses, g["losses"].tolist(), worst, report["__update_mismatch_fraction"][0]))


# ---------------------------------------------------------------------------------------------------
# block tail: bn + relu + tall conv + bn (+ residual) + relu as one autograd node with packed intermediates
# ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("cfg", [
    # in, hidden/out channels, conv_b kernel, top padding, residual, input (H, W), outer relu
    dict(cin=32, cout=32, k2=(9, 1), top=8, residual=True, hw=(41, 77), outer=True),      # 32-channel row-streaming kernels
    dict(cin=32, cout=32, k2=(16, 1), top=None, residual=False, hw=(70, 141), outer=False),
    dict(cin=32, cout=32, k2=(9, 1), top=8, residual=True, hw=(70, 141), outer=True),     # planes >= 2048: saved ReLU mask
    dict(cin=16, cout=128, k2=(6, 1), top=None, residual=True, hw=(30, 41), outer=True),  # 128-channel kernels
    dict(cin=32, cout=128, k2=(4, 1), top=3, residual=True, hw=(21, 133), outer=False),
    dict(cin=32, cout=32, k2=(9, 1), top=8, residual=True, hw=(41, 75), outer=True, node=False),   # odd width: unfused chain
])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_block_tail_node_matches_literal_modules(cpc, cfg, precision):
    """ScalogramEncoderBlock whose second conv runs on the row-streaming kernels: the single block-tail node (packed
    activations between bn_a and conv_b, packed dy between bn_b and conv_b) against the same block evaluated module by
    module (torch BatchNorm / ReLU, conv Functions) -- output, running statistics and every gradient.  In the bf16
    operand mode the node hands over the hi plane only; the literal chain rounds the same fp32 values to bf16 inside
    the conv calls, so the two agree far inside the mode's stated 1e-2 (bound here: 3e-3)."""
    cpc.ops.set_default_precision(precision)
    try:
        _block_tail_case(cpc, cfg, *((1e-4, TOL) if precision == "fp32" else (3e-3, 3e-3)))
    finally:
        cpc.ops.set_default_precision("fp32")


def _block_tail_case(cpc, cfg, out_tol, grad_tol):
    import copy
    block_cfg = {'in_channels': cfg['cin'], 'hidden_channels': None, 'out_channels': cfg['cout'], 'kernel_size_1': (3, 3),
                 'kernel_size_2': cfg['k2'], 'top_padding_1': None, 'top_padding_2': cfg['top'], 'padding_1': 0,
                 'padding_2': 0, 'stride_1': 2, 'stride_2': 1, 'pooling_1': 1, 'pooling_2': 1, 'bias': True,
                 'separable': False, 'residual': cfg['residual'], 'batch_norm': True, 'ceil_pooling': False}
    torch.manual_seed(12)
    block = cpc.ScalogramEncoderBlock(dict(block_cfg), name='b', activation_register=None).to(DEV).train()
    with torch.no_grad():
        for m in block.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.weight.uniform_(0.5, 1.5)
                m.bias.uniform_(-0.5, 0.5)
    ref_block = copy.deepcopy(block)
    gen = torch.Generator().manual_seed(13)
    x = torch.randn(3, cfg['cin'], *cfg['hw'], generator=gen).to(DEV)
    x1, x2 = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    y = block(x1, outer_relu=cfg['outer'])
    # the node must actually have been used (and must step aside for shapes it does not cover)
    assert type(y.grad_fn).__name__.startswith("_BlockTailFunction") == cfg.get('node', True), type(y.grad_fn).__name__
    with cpc.ops.second_order():                                   # literal module sequence
        y_ref = ref_block(x2, outer_relu=cfg['outer'])
    assert rel_err(y, y_ref) < out_tol
    gy = torch.randn(y.shape, generator=gen).to(DEV)
    (y * gy).sum().backward()
    (y_ref * gy).sum().backward()
    assert rel_err(x1.grad, x2.grad) < grad_tol
    noise_only = bn_shadowed_biases(block.state_dict().keys())
    for (n, p), (_, q) in zip(block.named_parameters(), ref_block.named_parameters()):
        if n in noise_only:
            assert float((p.grad - q.grad).abs().max()) < 1e-3 * float(gy.abs().sum()) ** 0.5, n   # both are rounding noise
        else:
            assert grad_err(p.grad, q.grad) < grad_tol, n
    for (n, b), (_, c) in zip(block.named_buffers(), ref_block.named_buffers()):
        assert rel_err(b.float(), c.float()) < out_tol, n
    # eval mode (validate()): running statistics, no autograd
    block.eval()
    ref_block.eval()
    with torch.no_grad():
        y_eval = block(x, outer_relu=cfg['outer'])
        with cpc.ops.second_order():
            y_eval_ref = ref_block(x, outer_relu=cfg['outer'])
    assert rel_err(y_eval, y_eval_ref) < out_tol


def test_activation_taps_receive_intermediates_and_match_the_fused_path(cpc):
    """With an ActivationRegister attached (audio_model.py:222-284) a block runs module by module so that the taps see
    the intermediate activations (SURVEY 8b); the result equals the block-tail node of the same block without taps."""
    import copy
    block_cfg = {'in_channels': 32, 'hidden_channels': None, 'out_channels': 32, 'kernel_size_1': (3, 3),
                 'kernel_size_2': (9, 1), 'top_padding_1': None, 'top_padding_2': 8, 'padding_1': 0, 'padding_2': 0,
                 'stride_1': 2, 'stride_2': 1, 'pooling_1': 1, 'pooling_2': 1, 'bias': True, 'separable': False,
                 'residual': True, 'batch_norm': True, 'ceil_pooling': False}
    torch.manual_seed(14)
    plain = cpc.ScalogramEncoderBlock(dict(block_cfg), name='blk', activation_register=None).to(DEV).train()
    register = cpc.ActivationRegister()
    tapped = cpc.ScalogramEncoderBlock(dict(block_cfg), name='blk', activation_register=register).to(DEV).train()
    tapped.load_state_dict(copy.deepcopy(plain.state_dict()))
    x = torch.randn(2, 32, 41, 77, generator=torch.Generator().manual_seed(15)).to(DEV)
    y_plain = plain(x.clone().requires_grad_(True), outer_relu=True)
    y_tapped = tapped(x.clone().requires_grad_(True), outer_relu=True)
    assert type(y_plain.grad_fn).__name__.startswith("_BlockTailFunction")
    assert not type(y_tapped.grad_fn).__name__.startswith("_BlockTailFunction")
    assert rel_err(y_tapped, y_plain) < 1e-4
    acts = register.get_activations()
    assert set(acts) == {'blk_main_conv_1', 'blk_main_conv_2'}
    assert tuple(acts['blk_main_conv_1'].shape) == (2, 32, 20, 38)          # after conv_a + bn + relu
    assert tuple(acts['blk_main_conv_2'].shape) == tuple(y_plain.shape)      # block output before the outer ReLU
    assert rel_err(torch.relu(acts['blk_main_conv_2']), y_plain) < 1e-4
    register.active = False
    register.activations.clear()
    tapped(x, outer_relu=True)
    assert len(register.get_activations()) == 0


# ---------------------------------------------------------------------------------------------------
# gradients through the front end, InverseCQT (SURVEY 8(f) row 3)
# ---------------------------------------------------------------------------------------------------

def test_trainable_cqt_gradients_match_reference_golden(cpc):
    """trainable_cqt=True / audio that requires grad: d<z, gz>/d(audio) and d/d(filters) of the CQT, and of the
    pooled phase scalogram, against the reference's autograd (constant_q_transform.py:155-172, scalogram_model.py:75-102)."""
    g = load_golden("cqt_grad.npz")
    kw = dict(sr=8000, fmin=55, n_bins=96, bins_per_octave=24, filter_scale=0.5, hop_length=64)
    cqt = cpc.CQT(trainable=True, **kw).to(DEV)
    assert list(cqt.conv_kernel_sizes) == list(g["kernel_sizes"])
    x = torch.from_numpy(g["x"]).to(DEV).requires_grad_(True)
    z = cqt(x)
    assert rel_err(z, g["z"]) < TOL
    (z * torch.from_numpy(g["gz"]).to(DEV)).sum().backward()
    assert rel_err(x.grad, g["gx"]) < TOL
    for i, conv in enumerate(cqt.conv_modules):
        assert rel_err(conv.weight.grad, g["gw%d" % i]) < TOL, i
    # frozen filters, differentiable input: same values through the same path
    frozen = cpc.CQT(trainable=False, **kw).to(DEV)
    x1 = torch.from_numpy(g["x"]).to(DEV).requires_grad_(True)
    (frozen(x1) * torch.from_numpy(g["gz"]).to(DEV)).sum().backward()
    assert rel_err(x1.grad, g["gx"]) < TOL
    assert all(c.weight.grad is None for c in frozen.conv_modules)
    # and the fused forward-only kernel agrees with the differentiable path
    with torch.no_grad():
        assert rel_err(frozen(x1), z.detach()) < TOL
    d = {'sample_rate': 8000, 'fmin': 55, 'n_bins': 96, 'bins_per_octave': 24, 'filter_scale': 0.5, 'hop_length': 64,
         'trainable_cqt': True}
    pre = cpc.PreprocessingModule(d, phase=True, offset_zero=True, output_power=1., pooling=[1, 2], scaling=3.).to(DEV)
    x2 = torch.from_numpy(g["x2"]).to(DEV).requires_grad_(True)
    y = pre(x2)
    assert y.grad_fn is not None
    assert rel_err(y[:, 0], g["y2"][:, 0]) < TOL
    (y * torch.from_numpy(g["gy2"]).to(DEV)).sum().backward()
    # 1/|z|^2 and 1/|z| factors make this gradient as ill-conditioned as the smallest coefficient: 5e-3
    assert rel_err(x2.grad, g["gx2"]) < 5 * TOL
    for i, conv in enumerate(pre.cqt.conv_modules):
        assert rel_err(conv.weight.grad, g["g2w%d" % i]) < 5 * TOL, i


def test_inverse_cqt_matches_reference_layers(cpc):
    """InverseCQT (constant_q_transform.py:180-260): the reference module's own ConvTranspose1d layers applied as its
    forward intends (fixture: oracle/make_golden.py golden_cqt_grad)."""
    g = load_golden("cqt_grad.npz")
    icqt = cpc.InverseCQT(sr=8000, fmin=55, n_bins=96, bins_per_octave=24, filter_scale=0.5, hop_length=64).to(DEV)
    assert [tuple(c.weight.shape) for c in icqt.conv_modules] == [(r.stop - r.start, 2, k) for r, k in
                                                                  zip(icqt.conv_index_ranges, icqt.conv_kernel_sizes)]
    z = torch.from_numpy(g["icqt_in"]).to(DEV).requires_grad_(True)
    out = icqt(z)
    assert tuple(out.shape) == g["icqt_out"].shape
    assert rel_err(out, g["icqt_out"]) < TOL
    # differentiable w.r.t. its input (dreaming optimises through it): compare with torch's conv_transpose1d
    gy = torch.randn(out.shape, generator=torch.Generator().manual_seed(8)).to(DEV)
    (gz,) = torch.autograd.grad((out * gy).sum(), z)
    z64 = z.detach().double().cpu().requires_grad_(True)
    res = 0
    for rng, k, conv in zip(icqt.conv_index_ranges, icqt.conv_kernel_sizes, icqt.conv_modules):
        band = z64[:, rng.start:rng.stop]
        band = band.permute(3, 0, 1, 2).reshape(2 * band.shape[0], band.shape[1], band.shape[2])
        res = res + F.conv_transpose1d(band, conv.weight.detach().double().cpu(), stride=64, padding=k // 2)
    res = res.view(2, z64.shape[0], 2, -1)
    ref = torch.stack([res[0, :, 0] - res[1, :, 0], res[0, :, 1] + res[1, :, 1]], dim=2)
    (gz_ref,) = torch.autograd.grad((ref * gy.double().cpu()).sum(), z64)
    assert rel_err(gz, gz_ref) < TOL


# ---------------------------------------------------------------------------------------------------
# Adam (cpc_adam_step) against torch.optim.Adam
# ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("weight_decay,maximize", [(0.0, False), (0.01, False), (0.0, True)])
def test_adam_matches_torch_adam(cpc, weight_decay, maximize):
    """Same parameters, same gradients, 25 steps: the single-kernel update against torch.optim.Adam (the optimizer the
    reference's trainer instantiates, contrastive_estimation_training.py:41,84).  Shapes cover the vector path, ragged
    tails, 1-element tensors, a 4-byte-aligned (not 16-byte-aligned) view and more tensors than one launch table holds."""
    gen = torch.Generator().manual_seed(3)
    shapes = [(512, 256, 5), (4097,), (1,), (3, 3), (32, 2, 3, 3), (8192,)] + [(17 + i,) for i in range(60)]
    base = [torch.randn(s, generator=gen) for s in shapes]
    backing = torch.zeros(1001, device=DEV)
    def make_params():
        ps = [b.clone().to(DEV).requires_grad_(True) for b in base]
        odd = backing.clone()[1:].detach()                       # data pointer is 4 mod 16
        odd.copy_(torch.arange(1000, device=DEV) * 1e-3)
        ps.append(odd.requires_grad_(True))
        return ps
    p_ref, p_new = make_params(), make_params()
    assert p_new[-1].data_ptr() % 16 == 4
    ref = torch.optim.Adam(p_ref, lr=3e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=weight_decay, maximize=maximize)
    new = cpc.optim.Adam(p_new, lr=3e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=weight_decay, maximize=maximize)
    for step in range(25):
        for a, b in zip(p_ref, p_new):
            g = torch.randn(a.shape, generator=gen).to(DEV) * (10.0 ** (step % 5 - 3))
            a.grad, b.grad = g.clone(), g.clone()
        ref.step()
        new.step()
    for a, b in zip(p_ref, p_new):
        assert torch.allclose(a, b, rtol=2e-6, atol=2e-7), float((a - b).abs().max())
    sa, sb = ref.state_dict(), new.state_dict()
    assert sa['state'].keys() == sb['state'].keys()
    for k in sa['state']:
        assert float(sb['state'][k]['step']) == float(sa['state'][k]['step']) == 25.0
        # moments: the lerp / fma roundings differ by an ulp of the largest term, so entries that cancel to ~0 only
        # agree absolutely (gradients reach 10, second moments 100)
        assert torch.allclose(sa['state'][k]['exp_avg'], sb['state'][k]['exp_avg'], rtol=1e-5, atol=1e-6), k
        assert torch.allclose(sa['state'][k]['exp_avg_sq'], sb['state'][k]['exp_avg_sq'], rtol=1e-5, atol=1e-9), k


def test_adam_state_dict_round_trip_and_flat_gradients(cpc):
    """(a) a torch.optim.Adam state_dict loads into cpc_b200.optim.Adam and training continues identically;
    (b) gradients read from a caller-provided flat buffer with grad_scale = 1/W equal averaged gradients."""
    gen = torch.Generator().manual_seed(4)
    base = [torch.randn(s, generator=gen) for s in [(300, 7), (129,), (64, 64)]]
    p_ref = [b.clone().to(DEV).requires_grad_(True) for b in base]
    p_new = [b.clone().to(DEV).requires_grad_(True) for b in base]
    ref = torch.optim.Adam(p_ref, lr=1e-2)
    def grads(ps):
        gs = [torch.randn(p.shape, generator=gen).to(DEV) for p in ps]
        return gs
    for _ in range(3):
        for p, g in zip(p_ref, grads(p_ref)):
            p.grad = g
        ref.step()
    with torch.no_grad():
        for a, b in zip(p_ref, p_new):
            b.copy_(a)
    new = cpc.optim.Adam(p_new, lr=1e-2)
    new.load_state_dict(copy.deepcopy(ref.state_dict()))        # (load_state_dict aliases same-device tensors)
    for _ in range(3):
        gs = grads(p_ref)
        for a, b, g in zip(p_ref, p_new, gs):
            a.grad = g.clone()
            b.grad = torch.zeros_like(g)                        # must be ignored: the flat views are the source
        flat = torch.cat([(4.0 * g).reshape(-1) for g in gs])    # "sum over 4 ranks"
        views, off = {}, 0
        for b, g in zip(p_new, gs):
            views[b] = flat[off:off + g.numel()].view_as(g)
            off += g.numel()
        ref.step()
        new.step(flat_grads=views, grad_scale=0.25)
    for a, b in zip(p_ref, p_new):
        assert torch.allclose(a, b, rtol=2e-6, atol=2e-7)
    assert float(new.state_dict()['state'][0]['step']) == 6.0


def test_two_rank_nccl_parity(cpc):
    """SURVEY 8e on hardware (needs two GPUs, skips otherwise): one process per GPU over NCCL, contiguous shards, per-GPU
    negatives; per-rank loss / gradients against the CPU oracle on that shard, averaged gradients against the mean of the
    per-shard oracle gradients, and the in-graph overlapped bucket all-reduce against the mean of per-rank gradients
    (tests/nccl_parity_worker.py)."""
    import os
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    worker = os.path.join(os.path.dirname(os.path.abspath(__file__)), "nccl_parity_worker.py")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29733", worker],
                         capture_output=True, text=True, timeout=300)
    print(out.stdout[-3000:])
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "RANK_OK 0" in out.stdout and "RANK_OK 1" in out.stdout


def test_bench_dump_outputs_of_the_last_timed_step(cpc, tmp_path):
    """bench.py --dump-outputs: loss, max score and gradients of the last timed step as float32, under 64 MB in all.
    Every timed step trains from the seeded initial state on batch i % 2, so the last steps of --steps 1 and --steps 3
    (both batch 0, separate runs) agree up to the rounding of one step, and that of --steps 2 (batch 1) does not."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dumps = {}
    for steps in (1, 3, 2):
        out_dir = tmp_path / str(steps)
        out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--workload", "raw_wave", "--batch", "2",
                              "--steps", str(steps), "--warmup", "1", "--dump-outputs", str(out_dir)],
                             capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, out.stderr[-3000:]
        assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == steps
        names = sorted(os.listdir(out_dir))
        assert names == ["gradients.npy", "loss.npy", "max_score.npy"], names
        assert sum(os.path.getsize(out_dir / n) for n in names) <= 64 << 20
        dumps[steps] = {n[:-4]: np.load(out_dir / n) for n in names}
    a, b, c = dumps[1], dumps[3], dumps[2]
    for name, v in a.items():
        assert v.dtype == np.float32 and np.isfinite(v).all(), name
    assert a["loss"].shape == () and a["gradients"].shape == (1 << 22,)
    assert float(np.abs(a["gradients"]).max()) > 0.0
    assert rel_err(b["loss"], a["loss"]) < 1e-5 and rel_err(b["max_score"], a["max_score"]) < 1e-5
    assert rel_err(b["gradients"], a["gradients"]) < 1e-3
    # at the initial weights the loss sits near chance for any white-noise batch: batch 1 moves it by only ~1e-4
    assert rel_err(c["loss"], a["loss"]) > 1e-5 and rel_err(c["gradients"], a["gradients"]) > 1e-2

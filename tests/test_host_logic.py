"""CPU tests: C-ABI library loads and exports every declared symbol, argument validation, host-side
module logic (geometry, state_dict layout, configs, sampler), and the data-parallel plumbing on gloo."""
import ctypes
import json
import os
import random
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import PKG, ROOT, load_golden


def test_library_exports_every_header_symbol(built_lib):
    header = open(os.path.join(ROOT, "include", "cpc_b200.h")).read()
    declared = set(re.findall(r"\b(cpc_[a-z0-9_]+)\s*\(", header))
    declared -= {"cpc_status"}
    from cpc_b200 import _lib
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    lib = ctypes.CDLL(built_lib)
    for name in declared:
        assert hasattr(lib, name), name
    lib = _lib.load()
    assert lib.cpc_abi_version() == _lib.ABI_VERSION
    assert lib.cpc_status_string(0) == b"ok" and lib.cpc_status_string(-1) == b"bad shape"


def test_abi_rejects_bad_arguments_before_touching_the_device(built_lib):
    from cpc_b200 import _lib
    lib = _lib.load()
    p = _lib.ConvParams()
    assert lib.cpc_conv_fwd(None, None, None, None, ctypes.byref(p), None, 0, None) == -1      # all-zero shape
    p.batch = p.c_in = p.h_in = p.w_in = p.c_out = p.h_out = p.w_out = p.kh = p.kw = p.stride_h = p.stride_w = 1
    assert lib.cpc_conv_fwd(None, None, None, None, ctypes.byref(p), None, 0, None) == -7      # null pointers
    p.stride_h = 0                                                                              # bad stride
    assert lib.cpc_conv_fwd(None, None, None, None, ctypes.byref(p), None, 0, None) == -1
    q = _lib.InfoNceParams()
    q.batch, q.steps, q.enc = 4, 100, 8
    assert lib.cpc_infonce_fwd(None, None, None, None, ctypes.byref(q), None, 0, None) == -6   # K > 64 unsupported
    c = _lib.CqtParams()
    c.batch, c.n_samples, c.x_pitch, c.n_bins, c.hop, c.n_frames, c.n_groups = 1, 100, 100, 4, 8, 2, 1
    c.kernel_size[0], c.bin_lo[0], c.bin_hi[0] = 128, 0, 4
    assert lib.cpc_cqt_fwd(None, None, None, None, None, ctypes.byref(c), None, 0, None) == -1  # frames overrun input
    assert lib.cpc_conv_fwd(None, None, None, None, None, None, 0, None) == -7
    b = _lib.BnParams()
    b.batch, b.channels, b.height, b.width, b.eps, b.training = 2, 3, 4, 6, 1e-5, 1
    assert lib.cpc_bn_packed_bytes(ctypes.byref(b)) == 2 * 2 * 3 * 4 * 8 * 2                   # two planes, pitch 8, bf16
    b.packed_planes = 1                                                                      # operand of a bf16-mode conv
    assert lib.cpc_bn_packed_bytes(ctypes.byref(b)) == 2 * 3 * 4 * 8 * 2
    b.packed_planes = 3
    assert lib.cpc_bn_packed_bytes(ctypes.byref(b)) == 0                                       # rejected by validation
    b.packed_planes = 0
    assert lib.cpc_bn_relu_fwd_packed(*([None] * 9), ctypes.byref(b), None, 0, None) == -7     # null pointers
    assert lib.cpc_bn_relu_bwd_packed(*([None] * 12), ctypes.byref(b), None, 0, None) == -7
    b.width = 0
    assert lib.cpc_bn_packed_bytes(ctypes.byref(b)) == 0                                       # bad shape
    assert lib.cpc_conv_pack_dy(None, None, None, ctypes.byref(p), None) == -1                 # stride 0 from above
    a = _lib.AdamParams(1e-3, 0.9, 0.999, 1e-8, 0.0, 1.0, 0)
    assert lib.cpc_adam_step(0, None, None, None, None, None, None, ctypes.byref(a), None) == -7  # no step counter
    a.beta2 = 1.5
    state = (ctypes.c_float * 4)()
    assert lib.cpc_adam_step(0, None, None, None, None, None, state, ctypes.byref(a), None) == -1  # beta out of range


def test_phase_accumulation_matches_reference_golden():
    """constant_q_transform.py:294-313 (plain tensor arithmetic, no kernel): values and state_dict keys."""
    import cpc_b200
    g = load_golden("cqt_grad.npz")
    acc = cpc_b200.PhaseAccumulation(sr=8000, fmin=55, n_bins=96, bins_per_octave=24, hop_length=64)
    assert set(acc.state_dict()) == {"scaling", "start_phase"}
    out = acc(torch.from_numpy(g["acc_in"]))
    want = torch.from_numpy(g["acc_out"])
    d = torch.remainder(out - want + np.pi, 2 * np.pi) - np.pi            # compare on the circle (mod 2 pi wrap)
    assert float(d.abs().max()) < 1e-4


def test_conv_dispatch_table_for_the_baseline_layers(built_lib):
    """Host-side dispatch (no device needed): which kernel family serves forward / dgrad / wgrad of every arch-7 conv at
    the BASELINE sizes, and the size of the canonical packed operands -- two dy replicas exactly for the strided convs
    whose data gradient reads column-shifted copies."""
    import cpc_b200
    from cpc_b200 import _lib
    lib = _lib.load()

    def params(ci, h, w, co, kh, kw, s, pt=0):
        p = _lib.ConvParams()
        p.batch, p.c_in, p.h_in, p.w_in, p.c_out, p.kh, p.kw = 64, ci, h, w, co, kh, kw
        p.stride_h = p.stride_w = s
        p.pad_top, p.pad_left, p.precision = pt, 0, 0
        p.h_out, p.w_out = (h + pt - kh) // s + 1, (w - kw) // s + 1
        return p

    def round8(v):
        return (v + 7) // 8 * 8

    table = {  # name: (params, families (fwd, dgrad, wgrad), dy replicas)
        "block0 conv_a": (params(2, 256, 629, 32, 3, 3, 2), (1, 1, 1), 0),      # C_in = 2: direct kernels for all three
        "block0 conv_b": (params(32, 127, 314, 32, 64, 1, 1, pt=63), (2, 2, 2), 1),
        "block1 conv_a": (params(32, 127, 314, 128, 3, 3, 2), (4, 4, 4), 2),
        "block1 conv_b": (params(128, 63, 156, 128, 30, 1, 1), (3, 3, 3), 1),
        "block1 residual": (params(32, 64, 157, 128, 1, 1, 1), (4, 4, 4), 1),
        "block2 conv_a": (params(128, 34, 156, 256, 3, 3, 2), (4, 4, 4), 2),
        "block2 conv_b": (params(256, 16, 77, 256, 15, 1, 1), (4, 4, 4), 1),
        "block3 conv_a": (params(256, 2, 77, 512, 2, 2, 1), (4, 4, 4), 1),
    }
    for name, (p, families, dy_rep) in table.items():
        got = tuple(lib.cpc_conv_kernel_family(ctypes.byref(p), which) for which in (0, 1, 2))
        assert got == families, (name, got)
        rows = 64 * p.c_out * p.h_out
        want = 0 if dy_rep == 0 else 2 * dy_rep * rows * round8(p.w_out + (1 if dy_rep == 2 else 0)) * 2
        assert lib.cpc_conv_packed_bytes(ctypes.byref(p), 1) == (want + 1023) // 1024 * 1024, name
        assert lib.cpc_conv_workspace_bytes(ctypes.byref(p), 1) >= 0
    # bf16 mode and the CUDA-core override change the answer
    p = table["block0 conv_b"][0]
    p.precision = 1                                                              # bf16 operand mode: same kernels, hi plane only
    assert [lib.cpc_conv_kernel_family(ctypes.byref(p), which) for which in (0, 1, 2)] == [2, 2, 2]
    rows = 64 * p.c_out * p.h_out
    assert lib.cpc_conv_packed_bytes(ctypes.byref(p), 1) == (rows * round8(p.w_out) * 2 + 1023) // 1024 * 1024
    p.precision = 0
    p.flags = _lib.CONV_FLAG_CUDA_CORE                                           # per-call switch in the struct: no global state
    assert lib.cpc_conv_kernel_family(ctypes.byref(p), 0) == 0
    assert lib.cpc_conv_packed_bytes(ctypes.byref(p), 1) == 0
    p.flags = _lib.CONV_FLAG_NO_TALL
    assert lib.cpc_conv_kernel_family(ctypes.byref(p), 0) == 4
    # ... and the environment is NOT consulted by the library (header: "no global state")
    p.flags = 0
    os.environ["CPC_FORCE_CUDA_CORE_CONV"] = "1"
    try:
        assert lib.cpc_conv_kernel_family(ctypes.byref(p), 0) == 2
        # the host mirror turns the same names into flags at call time
        assert cpc_b200.ops._conv_flags() & _lib.CONV_FLAG_CUDA_CORE
    finally:
        del os.environ["CPC_FORCE_CUDA_CORE_CONV"]
    assert cpc_b200.ops._conv_flags() == 0


def test_workspace_queries_cover_the_schedulers_and_the_per_step_regulariser(built_lib):
    """Host-side sizes (no device needed): the row-streaming conv kernels' workspace holds the packed operands plus the
    tile counter of their scheduler, also in the one-plane (bf16 operand) mode; the CUDA-core InfoNCE backward asks for
    the (R x C) sum buffer of the per-step regulariser and for nothing otherwise."""
    from cpc_b200 import _lib
    lib = _lib.load()
    p = _lib.ConvParams()
    p.batch, p.c_in, p.h_in, p.w_in, p.c_out, p.kh, p.kw = 4, 32, 127, 314, 32, 64, 1
    p.stride_h = p.stride_w = 1
    p.pad_top, p.h_out, p.w_out = 63, 127, 314

    def act(planes, h):
        return (planes * 4 * 32 * h * ((314 + 7) // 8 * 8) * 2 + 1023) // 1024 * 1024
    w_bytes = (64 * 32 * 64 * 2 + 1023) // 1024 * 1024
    for precision, planes in ((0, 2), (1, 1)):
        p.precision = precision
        assert lib.cpc_conv_kernel_family(ctypes.byref(p), 0) == 2
        assert lib.cpc_conv_workspace_bytes(ctypes.byref(p), 0) == act(planes, 127) + w_bytes + 256 + 1024
        assert lib.cpc_conv_workspace_bytes(ctypes.byref(p), 2) == 2 * act(planes, 127) + 1024
    q = _lib.InfoNceParams()
    q.batch, q.steps, q.enc, q.all_steps, q.score_kind, q.regularization = 8, 12, 512, 0, 1, 1.0
    assert lib.cpc_infonce_workspace_bytes(ctypes.byref(q), 1) == 8 * 8 * 4                 # per-step + regulariser
    q.regularization = 0.0
    assert lib.cpc_infonce_workspace_bytes(ctypes.byref(q), 1) == 0
    q.regularization, q.all_steps = 1.0, 1
    assert lib.cpc_infonce_workspace_bytes(ctypes.byref(q), 1) == 0                         # all-steps: sums stay in the tile
    fwd_reg = lib.cpc_infonce_workspace_bytes(ctypes.byref(q), 0)
    q.all_steps = 0
    assert lib.cpc_infonce_workspace_bytes(ctypes.byref(q), 0) >= 8 * 8 * 4 and fwd_reg > 0
    c = _lib.CqtParams()
    assert _lib.CQT_FLAG_HALF_OPERANDS == 2 and _lib.CQT_FLAG_NO_TENSOR == 1 and hasattr(c, "flags")


def test_weight_gradient_cta_hand_out(tmp_path):
    """umma.cuh: balance_group_ctas (pure host code, compiled here with nvcc and run on the CPU): the CTAs of a split-K
    weight-gradient launch are dealt to the accumulator groups so that atoms-per-CTA x cost-per-atom is level -- the arch-7
    64 x 1 layer's six tap groups (costs from its top padding) get 22 / 22 / 25 / 27 / 30 / 22 of the 148 SMs instead of 24
    each -- and degenerate inputs fall back (more groups than the table holds) or saturate (fewer atoms than CTAs)."""
    import shutil
    import subprocess
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    src = tmp_path / "hand_out.cu"
    src.write_text("""
#include <cstdio>
#include <cstdlib>
#include "umma.cuh"
int main(int argc, char** argv) {
    int n_units = atoi(argv[1]), total = atoi(argv[2]), n = argc - 3;
    int cost[256], start[cpc::umma::kMaxSplitGroups + 1];
    for (int g = 0; g < n; ++g) cost[g] = atoi(argv[3 + g]);
    int used = cpc::umma::balance_group_ctas(cost, n, n_units, total, start);
    printf("%d", used);
    for (int g = 0; used && g < n; ++g) printf(" %d", start[g + 1] - start[g]);
    printf("\\n");
    return 0;
}
""")
    exe = tmp_path / "hand_out"
    csrc = os.path.join(ROOT, "constrastive-predictive-coding-audio_b200", "csrc")
    inc = os.path.join(ROOT, "include")
    subprocess.run([nvcc, "-std=c++17", "-I", csrc, "-I", inc, "-o", str(exe), str(src), "-lcuda"], check=True,
                   capture_output=True)

    def run(n_units, total, *cost):
        out = subprocess.run([str(exe), str(n_units), str(total)] + [str(c) for c in cost], check=True,
                             capture_output=True, text=True).stdout.split()
        return [int(v) for v in out]

    got = run(320, 148, 64, 64, 69, 78, 87, 64)                  # e24 block 0 conv_b, B = 64: 320 pixel atoms
    assert got == [148, 22, 22, 25, 27, 30, 22]
    worst = max(-(-320 // c) * k for c, k in zip(got[1:], (64, 64, 69, 78, 87, 64)))
    assert worst == 960 and worst < 14 * 94                     # uniform split of the old kernel: 14 atoms x 94 blocks
    assert run(20, 148, 64, 64, 69, 78, 87, 64) == [120] + [20] * 6     # 20 atoms: one per CTA is the finest split
    assert run(192, 148, *([136] * 7 + [68])) == [148, 20, 20, 20, 20, 20, 20, 19, 9]
    assert run(100, 148, *([5] * 49)) == [0]                    # more groups than the table holds: caller keeps uniform
    assert run(100, 3, 1, 1, 1, 1) == [0]                       # fewer CTAs than groups


def test_second_order_switch_and_block_tail_gate():
    """ops.second_order() is a re-entrant context flag; the block-tail node never claims CPU tensors."""
    import cpc_b200
    ops = cpc_b200.ops
    assert not ops.second_order_enabled()
    with ops.second_order():
        assert ops.second_order_enabled()
        with ops.second_order(False):
            assert not ops.second_order_enabled()
        assert ops.second_order_enabled()
    assert not ops.second_order_enabled()
    conv = cpc_b200.Conv2d(32, 32, (9, 1))
    bn0, bn1 = torch.nn.BatchNorm2d(32), torch.nn.BatchNorm2d(32)
    assert not ops.block_tail_eligible(torch.zeros(1, 32, 20, 16), bn0, conv, 8, bn1)


def test_reference_snapshot_loads_without_reference_code(tmp_path):
    """A whole-model pickle written by the unmodified reference (tests/golden/ref_snapshot_1200, produced by
    oracle/make_golden.py golden_snapshot) is read without any reference module importable, and its state_dict loads
    strictly into the model this package builds from the same config dicts (setup_functions.py:134-164)."""
    import cpc_b200
    from conftest import GOLDEN
    from test_oracle_golden import small_resnet_blocks
    assert "audio_model" not in sys.modules and "scalogram_model" not in sys.modules
    path = os.path.join(GOLDEN, "ref_snapshot_1200")
    want = load_golden("ref_snapshot_state.npz")
    state = cpc_b200.snapshots.extract_state_dict(path)
    assert list(state) == list(want) or set(state) == set(want)
    for k, v in state.items():
        assert np.array_equal(v.numpy(), want[k]), k
    blocks = small_resnet_blocks()
    blocks[0]['in_channels'] = 1
    blocks[2] = dict(blocks[2], kernel_size_1=(30, 2), pooling_1=1, ceil_pooling=False)
    blocks[1] = dict(blocks[1], kernel_size_2=(35, 1))
    pre = cpc_b200.PreprocessingModule(dict(cpc_b200.cqt_default_dict), phase=True)
    enc = cpc_b200.ScalogramResidualEncoder({'phase': True, 'blocks': blocks, 'activation_register': None},
                                            preprocessing_module=pre)
    ar = cpc_b200.ConvolutionalArModel({'kernel_sizes': [3, 3], 'channel_count': [24, 16, 16], 'stride': [1, 1],
                                        'pooling': [1, 2], 'bias': True, 'batch_norm': True, 'residual': False,
                                        'activation_register': None})
    model = cpc_b200.AudioPredictiveCodingModel(enc, ar, enc_size=24, ar_size=16, visible_steps=10, prediction_steps=3)
    assert cpc_b200.snapshots.load_reference_snapshot(model, path, strict=True) == 1200
    for k, v in model.state_dict().items():
        assert np.array_equal(v.numpy(), want[k]), k
    # round trip through the portable form
    out = tmp_path / "mine_7"
    cpc_b200.snapshots.save_snapshot(model, str(out))
    again = cpc_b200.snapshots.extract_state_dict(str(out))
    assert set(again) == set(want) and cpc_b200.snapshots.snapshot_step(str(out)) == 7
    # the stand-ins are inert: calling one explains what to do instead of computing anything
    graph = cpc_b200.snapshots.read_reference_snapshot(path)
    with pytest.raises(RuntimeError):
        graph(torch.zeros(1, 1, 8))
    # a pickle may name any callable: globals outside the reference / torch / container set are refused
    import pickle

    class Hostile:
        def __reduce__(self):
            return (os.getcwd, ())
    bad = tmp_path / "bad_1"
    bad.write_bytes(pickle.dumps(Hostile()))
    with pytest.raises(pickle.UnpicklingError):
        cpc_b200.snapshots.read_reference_snapshot(str(bad))


def test_no_cpu_fallback(built_lib):
    import cpc_b200
    enc = cpc_b200.AudioEncoder()
    with pytest.raises(cpc_b200._lib.CpcError):
        enc(torch.zeros(1, 1, 2000))
    with pytest.raises(cpc_b200._lib.CpcError):
        cpc_b200.ops.infonce(torch.zeros(2, 2, 4), torch.zeros(2, 4, 2), True)
    with pytest.raises(cpc_b200._lib.CpcError):
        cpc_b200.CQT(filter_scale=0.5)(torch.zeros(1, 1, 20000))
    with pytest.raises(cpc_b200._lib.CpcError):                           # differentiable path: same rule
        cpc_b200.CQT(filter_scale=0.5, trainable=True)(torch.zeros(1, 1, 20000))
    p = torch.nn.Parameter(torch.zeros(8))
    p.grad = torch.zeros(8)
    with pytest.raises(cpc_b200._lib.CpcError):
        cpc_b200.optim.Adam([p]).step()


def test_audio_encoder_known_answers():
    import cpc_b200
    enc = cpc_b200.AudioEncoder({'strides': [5, 4, 2, 2, 2], 'kernel_sizes': [10, 8, 4, 4, 4],
                                 'channel_count': [32] * 5, 'bias': True})
    assert enc.downsampling_factor == 160 and enc.receptive_field == 465       # tests/test_audioEncoder.py
    g = load_golden("audio_encoder.npz")
    assert list(g["kat_rf_ds"]) == [enc.receptive_field, enc.downsampling_factor]


def test_cqt_module_layout_matches_reference_golden():
    import cpc_b200
    cqt = cpc_b200.CQT(sr=16000, fmin=30, n_bins=256, bins_per_octave=32, filter_scale=0.5, hop_length=128)
    assert cqt.conv_kernel_sizes == [16384, 8192, 4096, 2048, 1024, 512, 256, 128, 64]
    assert [(r.start, r.stop) for r in cqt.conv_index_ranges][:3] == [(0, 19), (19, 51), (51, 83)]
    assert [tuple(c.weight.shape) for c in cqt.conv_modules][:2] == [(38, 1, 16384), (64, 1, 8192)]
    assert not any(p.requires_grad for p in cqt.parameters())
    assert sum(p.numel() for p in cqt.parameters()) == 1664640
    plan = cqt.kernel_plan()
    assert plan["weight_offsets"][1] == 38 * 16384
    g = load_golden("cqt.npz")
    cqt2 = cpc_b200.CQT(sr=8000, fmin=55, n_bins=120, bins_per_octave=24, filter_scale=1., hop_length=64)
    assert cqt2.conv_kernel_sizes == list(g["kernel_sizes2"])
    # the product's own filterbank construction agrees with the oracle's restatement
    import cpc_oracle as O
    ref = O.CqtPlan(16000, 30, 256, 32, 0.5, 128)
    for w, conv in zip(ref.weights, cqt.conv_modules):
        assert np.array_equal(w, conv.weight[:, 0].numpy())


def test_configs_equal_reference_as_imported():
    from cpc_b200 import configs
    ref = load_golden("configs.json")

    def clean(v):
        if isinstance(v, dict):
            return {k: clean(x) for k, x in v.items()}
        if isinstance(v, (list, tuple)):
            return [clean(x) for x in v]
        if isinstance(v, (int, float, str, bool)) or v is None:
            return v
        return getattr(v, "__name__", str(v))

    for name in ("e24", "e25", "e20"):
        mine = clean(configs.experiment(name))
        theirs = ref[name]
        if name == "e20":                      # the gradient penalty is not implemented on the B200 path yet
            theirs["training_config"]["wasserstein_gradient_penalty"] = False
        assert mine == theirs, name


def test_model_geometry_and_state_dict_keys():
    from cpc_b200 import configs
    e = configs.experiment("e24")
    model, pre, _ = configs.setup_model(e["cqt_config"], e["encoder_config"], e["ar_model_config"],
                                        e["training_config"])
    assert model.item_length == 97024 and model.encoder.receptive_field == 19200
    assert model.encoder.downsampling_factor == 1024
    assert model.parameter_count() == 9324864
    g = load_golden("trainer_cqt.npz")
    ref_keys = {k[3:] for k in g if k.startswith("s0.")}
    assert any(k.startswith("encoder.blocks.0.main_modules.") for k in ref_keys)
    assert pre.receptive_field == 16384 and pre.downsampling_factor == 128


def test_file_batch_sampler_bit_exact():
    from cpc_b200 import FileBatchSampler
    for c in load_golden("sampler.json"):
        if c["global_seed"] is not None:
            random.seed(c["global_seed"])
        s = FileBatchSampler(c["counts"], c["batch_size"], c["file_batch_size"], drop_last=True, seed=c["seed"])
        assert len(s) == c["len"]
        epochs = [[list(b) for b in iter(s)] for _ in range(2)]
        assert epochs == c["epochs"], c


def test_shard_batch_is_dataparallel_chunking():
    from cpc_b200 import ddp
    x = torch.arange(24).view(8, 3)
    assert torch.equal(torch.cat([ddp.shard_batch(x, r, 4) for r in range(4)]), x)
    assert torch.equal(ddp.shard_batch(x, 1, 4), x[2:4])
    with pytest.raises(ValueError):
        ddp.shard_batch(x, 0, 3)


WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from cpc_b200 import ddp
rank, world, _ = ddp.init_from_env("gloo")
torch.manual_seed(0)
model = torch.nn.Sequential(torch.nn.Linear(16, 32), torch.nn.ReLU(), torch.nn.Linear(32, 8), torch.nn.Linear(8, 4))
if rank == 1:
    for p in model.parameters():
        p.data.add_(1.0)
ddp.broadcast_parameters(model, 0)
red = ddp.GradientBucketReducer(model, bucket_mb=0.0005)
assert len(red.buckets) >= 2
g = torch.Generator().manual_seed(7)
x = torch.randn(8, 16, generator=g)
y = torch.randn(8, 4, generator=g)
mine = ddp.shard_batch(x, rank, world), ddp.shard_batch(y, rank, world)
loss = ((model(mine[0]) - mine[1]) ** 2).mean()
loss.backward()
launched = red.launched_during_backward
red.finish()
# single-process reference: mean over ranks of per-shard gradients
ref = torch.nn.Sequential(torch.nn.Linear(16, 32), torch.nn.ReLU(), torch.nn.Linear(32, 8), torch.nn.Linear(8, 4))
ref.load_state_dict(model.state_dict())
total = 0
for r in range(world):
    total = total + ((ref(ddp.shard_batch(x, r, world)) - ddp.shard_batch(y, r, world)) ** 2).mean() / world
total.backward()
for p, q in zip(model.parameters(), ref.parameters()):
    assert torch.allclose(p.grad, q.grad, atol=1e-6), (p.grad - q.grad).abs().max()
assert launched == len(red.buckets), (launched, len(red.buckets))
# the synchronous helper used around CUDA-graph replays gives the same averages
red.remove()
model.zero_grad(set_to_none=True)
loss = ((model(mine[0]) - mine[1]) ** 2).mean()
loss.backward()
ddp.allreduce_gradients([p for p in model.parameters()], world, bucket_mb=0.0005)
for p, q in zip(model.parameters(), ref.parameters()):
    assert torch.allclose(p.grad, q.grad, atol=1e-6), (p.grad - q.grad).abs().max()
# ShardedBatchSampler: every rank sees rank 0's batches (drawn from rank 0's unseeded global `random`), takes its slice
import random
from cpc_b200.sampler import FileBatchSampler
random.seed(100 + rank)                                      # ranks deliberately start from different random states
base = FileBatchSampler([24], batch_size=8, file_batch_size=1, drop_last=True)
if rank == 0:
    random.seed(100)
    expect = [list(b) for b in FileBatchSampler([24], batch_size=8, file_batch_size=1, drop_last=True)]
    random.seed(100)
else:
    expect = None
box = [expect]
dist.broadcast_object_list(box, src=0)
expect = box[0]
mine = list(ddp.ShardedBatchSampler(base, rank, world))
assert mine == [b[rank * 4:(rank + 1) * 4] for b in expect], (mine, expect)
# a NaN on one rank makes every rank leave train() before the optimizer touches the weights
import cpc_b200
class Toy(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.w = torch.nn.Parameter(torch.ones(3))
    def forward(self, batch):
        return self.w, batch
class ToyTrainer(cpc_b200.ContrastiveEstimationTrainer):
    def loss_on_batch(self, batch):
        loss = (self.model.w ** 2).sum() * (float("nan") if self.rank == 1 else 1.0)
        return loss, loss.detach()
class Items(torch.utils.data.Dataset):
    def __len__(self): return 16
    def __getitem__(self, i): return torch.zeros(4)
    def get_example_count_per_file(self): return [16]
toy = Toy()
trainer = ToyTrainer(model=toy, dataset=Items(), device=torch.device("cpu"), optimizer=torch.optim.SGD, verbose=False)
out = trainer.train(batch_size=8, epochs=1, lr=0.1, num_workers=0, max_steps=3)
assert out is None and trainer.training_step == 0 and bool((toy.w == 1).all()), (trainer.training_step, toy.w)
dist.barrier()
print("RANK_OK", rank)
'''


def test_gradient_bucket_reducer_gloo_world2(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29671", WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, str(script), PKG], env=dict(env, RANK=str(r), LOCAL_RANK=str(r)),
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and "RANK_OK %d" % r in o, o


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver times next to ours): exactly one JSON line on stdout with the
    contract's keys, the same metric / unit / workload as our arm, and no work on ranks other than 0."""
    env = dict(os.environ, OMP_NUM_THREADS="4")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    line = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["metric"] == "train audio-sec/sec" and line["unit"] == "audio-s/s"
    assert line["vs_baseline"] is None and line["higher_is_better"] is True and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "e24" in line["config"]["workload"]
    # a non-zero rank of a torchrun launch exits 0 without output
    quiet = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                           capture_output=True, text=True, timeout=120, env=dict(env, RANK="1", WORLD_SIZE="2"))
    assert quiet.returncode == 0 and quiet.stdout.strip() == ""
    # our arm refuses to run without a GPU instead of falling back
    if not torch.cuda.is_available():
        ours = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True,
                              timeout=300, env=env)
        assert ours.returncode != 0 and "no CPU fallback" in (ours.stderr + ours.stdout)
    # --dump-outputs is refused where there is no timed training step of ours to dump
    refused = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs",
                              "unused"], capture_output=True, text=True, timeout=120, env=env)
    assert refused.returncode != 0 and "--dump-outputs" in refused.stderr and refused.stdout.strip() == ""


def test_bench_dump_outputs_writes_float32_and_a_fixed_sample_of_long_arrays(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 1000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"loss": torch.tensor(1.5, dtype=torch.float64),
                                               "parameters": torch.arange(5000, dtype=torch.float64).view(50, 100)})
    loss = np.load(tmp_path / "a" / "loss.npy")
    assert loss.dtype == np.float32 and loss.shape == () and float(loss) == 1.5
    a, b = np.load(tmp_path / "a" / "parameters.npy"), np.load(tmp_path / "b" / "parameters.npy")
    assert a.dtype == np.float32 and a.shape == (1000,)
    assert np.array_equal(a, b)                                   # the same entries on every run
    assert bool((np.diff(a) > 0).all()) and a[0] >= 0 and a[-1] < 5000   # distinct entries, in index order


def test_literal_loss_block_and_small_helpers():
    """Host-side pieces that never touch a kernel: the literal loss block used for score functions the fused kernel
    does not know (contrastive_estimation_training.py:108-122,141) against the oracle, DeterministicSampler (:363-382),
    num_parameters (audio_model.py:293-297)."""
    import cpc_b200
    import cpc_oracle as O
    from cpc_b200.trainer import reference_loss_from_scores
    gen = torch.Generator().manual_seed(3)
    pred = torch.randn(5, 4, 16, generator=gen) * 0.3
    tgt = torch.randn(5, 16, 4, generator=gen)
    for fn, kind in ((cpc_b200.linear_score_function, "linear"), (cpc_b200.softplus_score_function, "softplus")):
        for all_steps in (True, False):
            loss, mx = reference_loss_from_scores(fn(pred, tgt), 5, 4, all_steps, 0.3)
            want, want_mx = O.infonce_loss(pred, tgt, all_steps, kind, 0.3)
            assert abs(float(loss) - float(want)) < 1e-6 * max(1.0, abs(float(want))), (kind, all_steps)
            assert abs(float(mx) - float(want_mx)) < 1e-6
    # the inverse-square-distance score (:25-33) keeps its (B, K, B, K) contract
    assert tuple(cpc_b200.difference_score_function(pred, tgt).shape) == (5, 4, 5, 4)
    # DeterministicSampler (:363-382): single indices, shuffled by random.seed(seed), the same order on every pass
    import random
    sampler = cpc_b200.DeterministicSampler(list(range(10)), seed=3)
    want = list(range(10))
    random.seed(3)
    random.shuffle(want)
    assert list(sampler) == want and list(sampler) == want and len(sampler) == 10 and want != list(range(10))
    assert list(cpc_b200.DeterministicSampler(list(range(10)))) == list(cpc_b200.DeterministicSampler(list(range(10)), seed=0))
    enc = cpc_b200.AudioEncoder()
    assert cpc_b200.num_parameters(enc) == sum(p.numel() for p in enc.parameters())
    assert enc.receptive_field == 465 and enc.downsampling_factor == 160


def test_gru_model_fused_sequence_call_equals_the_unrolled_cells():
    """AudioGRUModel (audio_model.py:47-77): the single fused library call over the whole sequence (the CUDA path; on the
    CPU torch's native kernel behind the same entry point) computes exactly the unrolled nn.GRUCell loop of the reference
    -- last hidden state, input and parameter gradients, with and without biases, with a persistent hidden state."""
    import copy
    import torch
    from cpc_b200 import ar_models
    torch.manual_seed(0)
    for bias in (True, False):
        fused = ar_models.AudioGRUModel(12, 7, bias=bias).double()
        loop = copy.deepcopy(fused)
        fused.fused, loop.fused = True, False
        assert set(fused.state_dict()) == ({"gruCell.weight_ih", "gruCell.weight_hh", "gruCell.bias_ih", "gruCell.bias_hh"}
                                           if bias else {"gruCell.weight_ih", "gruCell.weight_hh"})
        x = torch.randn(5, 12, 9, dtype=torch.double)
        xa, xb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
        ya, yb = fused(xa), loop(xb)
        assert float((ya - yb).abs().max()) < 1e-12
        g = torch.randn_like(ya)
        (ya * g).sum().backward()
        (yb * g).sum().backward()
        assert float((xa.grad - xb.grad).abs().max()) < 1e-12
        for p_, q_ in zip(fused.parameters(), loop.parameters()):
            assert float((p_.grad - q_.grad).abs().max()) < 1e-12
    fused = ar_models.AudioGRUModel(12, 7, reset_hidden=False)
    loop = copy.deepcopy(fused)
    fused.fused, loop.fused = True, False
    x = torch.randn(5, 12, 9)
    for _ in range(2):                                              # the second call starts from the kept state
        ya, yb = fused(x), loop(x)
        fused.hidden, loop.hidden = fused.hidden.detach(), loop.hidden.detach()
    assert float((ya - yb).abs().max()) < 1e-6
    assert ar_models.AudioGRUModel(12, 7)._use_fused(x) is False    # CPU tensors keep the stock loop by default


def test_preprocessing_identity_and_geometry_without_kernels():
    """PreprocessingModule(cqt_dict=None) is the identity (scalogram_model.py:77-78); with a CQT its geometry attributes
    follow the filterbank (:48-51, :70-72); unsupported scalogram pooling is refused at construction time."""
    import cpc_b200
    pre = cpc_b200.PreprocessingModule(None)
    x = torch.randn(2, 1, 50)
    assert pre(x) is x and pre.downsampling_factor == 1 and pre.receptive_field == 1
    d = dict(cpc_b200.cqt_default_dict)
    pre = cpc_b200.PreprocessingModule(d, phase=True, pooling=[1, 2])
    assert pre.receptive_field == 16384 and pre.downsampling_factor == 256
    assert sorted(k for k in pre.state_dict() if not k.startswith("cqt.")) == ["phase_diff.fixed_phase_diff", "phase_diff.scaling"]
    assert len(pre.cqt.conv_modules) == 9 and pre.cqt.conv_modules[0].weight.shape == (38, 1, 16384)
    assert not any(p.requires_grad for p in pre.parameters())
    pre.cqt.trainable = True
    assert all(p.requires_grad for p in pre.cqt.parameters()) and pre.cqt.needs_autograd(x)
    with torch.no_grad():
        assert not pre.cqt.needs_autograd(x)
    with pytest.raises(NotImplementedError):
        cpc_b200.PreprocessingModule(d, pooling=[2, 2])


def test_audio_dataset_matches_reference_index_logic(tmp_path):
    """AudioDataset / AudioTestingDataset (audio_dataset.py:16-199; SURVEY 8f-4) on real WAV files against the reference's
    own index arithmetic and cross-file item assembly (tests/golden/audio_dataset.json: the reference classes with only the
    decoder stubbed, oracle/make_golden.py::golden_audio_dataset), plus the native PCM reader and FileBatchSampler on top."""
    import wave
    import cpc_b200
    g = load_golden("audio_dataset.json")
    names = [n for n, _ in g["files"]]
    lengths = dict((n, l) for n, l in g["files"])

    def pcm(k, pos):                                             # int16 content of file k at position pos
        return ((np.asarray(pos, dtype=np.int64) * 7 + k * 1000) % 30000 - 15000).astype(np.int16)

    for k, (name, n) in enumerate(g["files"]):
        path = tmp_path / name
        path.parent.mkdir(parents=True, exist_ok=True)
        with wave.open(str(path), "wb") as fh:
            fh.setnchannels(2)
            fh.setsampwidth(2)
            fh.setframerate(16000)
            stereo = np.stack([pcm(k, np.arange(n)), np.zeros(n, dtype=np.int16)], axis=1)   # channel 0 is what is read
            fh.writeframes(stereo.tobytes())
    for case in g["cases"]:
        ds = getattr(cpc_b200, case["class"])(str(tmp_path), item_length=case["item_length"], unique_length=case["unique_length"])
        order = [os.path.relpath(str(f), str(tmp_path)).replace(os.sep, "/") for f in ds.files]
        assert order == case["order"]
        assert [int(v) for v in ds.start_samples] == case["start_samples"]
        assert len(ds) == case["len"] and [int(v) for v in ds.get_example_count_per_file()] == case["counts"]
        for idx, want in case["items"].items():
            item = ds[int(idx)]
            if case["class"] == "AudioTestingDataset":
                item, label = item
                assert int(label) == want["label"]
            assert item.dtype == torch.float32 and item.numel() == want["n"] == case["item_length"]
            # rebuild the (file, position) sequence the reference read: runs of consecutive positions, a new file at a break
            k, pos = divmod(want["first"], 100000)
            expect, at, total = [], 0, 0
            for brk in want["breaks"] + [want["n"] - 1]:
                count = brk + 1 - at
                expect.append(pcm(k, pos + np.arange(count)))
                total += int((k * 100000 + pos + np.arange(count)).sum())
                if brk != want["n"] - 1:
                    k, pos, at = names.index(order[order.index(names[k]) + 1]), 0, brk + 1
            assert total == want["sum"]
            assert np.array_equal(item.numpy(), np.concatenate(expect).astype(np.float32) / 32768.0), (case["class"], idx)
    # the sampler the trainer puts on top consumes the per-file counts
    ds = cpc_b200.AudioDataset(str(tmp_path), item_length=1000, unique_length=400)
    batches = list(cpc_b200.FileBatchSampler(ds.get_example_count_per_file(), batch_size=8, file_batch_size=4, seed=0))
    assert batches and all(len(b) == 8 and max(b) < len(ds) for b in batches)
    ds.dummy_load = True
    assert ds[0].shape[0] == 1000
    assert lengths["d_last.wav"] == 300 and cpc_b200.audio_dataset.read_wav(tmp_path / "d_last.wav", 5, 298).numel() == 2


def test_snapshot_unpickler_refuses_globals_outside_the_allow_list():
    """A snapshot may only name reference classes (stand-ins) and an exact list of torch / numpy / container globals:
    `getattr`, re-exported modules under the torch root (torch.serialization.os) and arbitrary torch callables are refused."""
    import io
    import pickle
    from cpc_b200 import snapshots
    for payload in (b"cbuiltins\ngetattr\n.", b"ctorch.serialization\nos\n.", b"ctorch.hub\nload\n.",
                    b"ctorch.utils.cpp_extension\nload\n.", b"cos\nsystem\n.", b"ctorch.nn.modules.module\n_addindent\n."):
        with pytest.raises(pickle.UnpicklingError):
            snapshots._SnapshotUnpickler(io.BytesIO(payload)).load()
    assert snapshots._SnapshotUnpickler(io.BytesIO(b"ccollections\nOrderedDict\n.")).load() is __import__("collections").OrderedDict
    assert snapshots._SnapshotUnpickler(io.BytesIO(b"ctorch.nn.modules.conv\nConv2d\n.")).load() is torch.nn.Conv2d
    stub = snapshots._SnapshotUnpickler(io.BytesIO(b"caudio_model\nAudioEncoder\n.")).load()
    assert issubclass(stub, torch.nn.Module) and stub.__name__ == "AudioEncoder"

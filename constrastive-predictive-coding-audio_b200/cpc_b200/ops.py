"""torch.autograd.Function wrappers around the C-ABI kernels.

PyTorch is plumbing here: it owns the device buffers and the stream; all arithmetic happens inside
libcpc_b200.so.  Every op raises on non-CUDA tensors -- there is no CPU path.
"""
import contextlib
import ctypes

import torch
from torch.autograd.function import once_differentiable

from . import _lib

_PRECISION = {"fp32": 0, "bf16": 1}
_default_precision = "fp32"


def set_default_precision(name):
    """'fp32' (fp32-faithful, the parity mode) or 'bf16' (bf16 operands, fp32 accumulate)."""
    global _default_precision
    if name not in _PRECISION:
        raise ValueError(name)
    _default_precision = name


def get_default_precision():
    return _default_precision


def strict_fp32_libraries():
    """The stock-PyTorch parts of the step (AR model convs / attention, the W_k Linear) run on cuDNN / cuBLAS; both
    would otherwise be free to use TF32 (10-bit mantissa) while the result is reported as fp32 and compared with the
    reference's CPU fp32.  Called by the trainer and setup_model in the fp32 parity mode."""
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


# Second-order mode (the Wasserstein gradient penalty, contrastive_estimation_training.py:144-155, differentiates
# d(sum scores)/d(scalogram) once more): convolutions stay on the B200 kernels -- their backward is then recorded
# as differentiable dgrad / wgrad Functions -- while the fused BN+ReLU and max-pool Functions, whose backward
# kernels have no second derivative, step aside for the literal module sequence.
_second_order = False


@contextlib.contextmanager
def second_order(enabled=True):
    global _second_order
    previous, _second_order = _second_order, bool(enabled)
    try:
        yield
    finally:
        _second_order = previous


def second_order_enabled():
    return _second_order


# Kernel-selection switches (A/B tests, diagnostics).  The C-ABI library itself holds no state and reads no
# environment: each call receives the switches in its parameter struct's ``flags`` field.  On the host side they
# can be set programmatically (``ops.kernel_switches["CPC_NO_TENSOR_CQT"] = True``) or through environment
# variables of the same names, read at call time.
kernel_switches = {}
_CONV_SWITCHES = (("CPC_FORCE_CUDA_CORE_CONV", _lib.CONV_FLAG_CUDA_CORE), ("CPC_NO_TALL_CONV", _lib.CONV_FLAG_NO_TALL),
                  ("CPC_NO_SMALLK_CONV", _lib.CONV_FLAG_NO_SMALLK), ("CPC_NO_FUSED_DGRAD", _lib.CONV_FLAG_NO_FUSED_DGRAD),
                  ("CPC_NO_MMA_SMALL_WGRAD", _lib.CONV_FLAG_NO_MMA_SMALL_WGRAD))


def _switch(name):
    import os
    if name in kernel_switches:
        return bool(kernel_switches[name])
    return os.environ.get(name) == "1"


switch = _switch


def _conv_flags():
    flags = 0
    for name, bit in _CONV_SWITCHES:
        if _switch(name):
            flags |= bit
    return flags


def _require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise _lib.CpcError("cpc_b200 ops need CUDA tensors on a B200 (sm_100a); got a %s tensor and there is "
                                "no CPU fallback" % t.device.type)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


class KernelProfiler:
    """Brackets every C-ABI call with CUDA events on the launching stream while active (bench.py uses it
    to time the dominant kernel inside real training steps).  ``summary()`` synchronises and returns the
    per-(op, shape) totals sorted by time."""

    def __init__(self):
        self.records = []

    def __enter__(self):
        global _profiler
        _profiler = self
        return self

    def __exit__(self, *exc):
        global _profiler
        _profiler = None

    def summary(self):
        torch.cuda.synchronize()
        agg = {}
        for key, flops, nbytes, e0, e1 in self.records:
            a = agg.setdefault(key, {"key": key, "count": 0, "total_ms": 0.0, "flops_per_launch": flops,
                                     "bytes_per_launch": nbytes})
            a["count"] += 1
            a["total_ms"] += e0.elapsed_time(e1)
        total = sum(a["total_ms"] for a in agg.values()) or 1.0
        out = sorted(agg.values(), key=lambda a: -a["total_ms"])
        for a in out:
            a["avg_ms"] = a["total_ms"] / a["count"]
            a["share"] = a["total_ms"] / total
            a["tflops"] = a["flops_per_launch"] / (a["avg_ms"] * 1e-3) / 1e12 if a["avg_ms"] > 0 else 0.0
            a["gbs"] = a["bytes_per_launch"] / (a["avg_ms"] * 1e-3) / 1e9 if a["avg_ms"] > 0 else 0.0
        return out


_profiler = None


def _call(key, flops, fn, *args, nbytes=0.0):
    """Invoke one C-ABI entry point (optionally event-timed) and raise on a non-zero status.  ``flops`` /
    ``nbytes`` are the ALGORITHMIC work of the call (what the roofline fractions are computed from)."""
    if _profiler is None:
        status = fn(*args)
    else:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        status = fn(*args)
        e1.record()
        _profiler.records.append((key, flops, nbytes, e0, e1))
    _lib.check(status, key.split(" ")[0])


CONV_FAMILIES = {0: "conv_tiled_cuda_core", 1: "conv_small_k_direct", 2: "tall_conv_tcgen05_32ch", 3: "tall_conv_tcgen05_128ch",
                 4: "conv_implicit_gemm_tcgen05"}


def _conv_key(tag, p):
    which = {"cpc_conv_fwd": 0, "cpc_conv_dgrad": 1, "cpc_conv_wgrad": 2}[tag]
    fam = CONV_FAMILIES.get(_lib.load().cpc_conv_kernel_family(ctypes.byref(p), which), "?")
    return "%s b%d %dx%dx%d->%dx%dx%d k%dx%d s%dx%d [%s]" % (tag, p.batch, p.c_in, p.h_in, p.w_in, p.c_out, p.h_out,
                                                            p.w_out, p.kh, p.kw, p.stride_h, p.stride_w, fam)


def _conv_flops(p):
    return 2.0 * p.c_out * p.c_in * p.kh * p.kw * p.batch * p.h_out * p.w_out


def _workspace(nbytes, device):
    if nbytes == 0:
        return None
    return torch.empty(int(nbytes), dtype=torch.uint8, device=device)


# --------------------------------------------------------------------------------------------------
# convolution
# --------------------------------------------------------------------------------------------------

_OVERLAP_MAX_FLOPS = 60e9                                     # ~0.15 ms at the generic kernel's rate
_side_streams = {}


def _side_stream(device):
    key = (device.type, device.index)
    if key not in _side_streams:
        _side_streams[key] = torch.cuda.Stream(device=device)
    return _side_streams[key]


def _conv_params(x_shape, w_shape, stride, pad_top, pad_left, out_hw, relu, precision):
    p = _lib.ConvParams()
    p.batch, p.c_in, p.h_in, p.w_in = x_shape
    p.c_out, _, p.kh, p.kw = w_shape
    p.h_out, p.w_out = out_hw
    p.stride_h, p.stride_w = stride
    p.pad_top, p.pad_left = pad_top, pad_left
    p.relu = int(relu)
    p.precision = _PRECISION[precision]
    p.flags = _conv_flags()
    return p


def _pack_operand(lib, t, p, operand):
    """bf16 hi/lo planes of a conv operand, packed once for every kernel that reads it (None when the
    configuration has no tensor-core kernel that would use them)."""
    nbytes = lib.cpc_conv_packed_bytes(ctypes.byref(p), operand)
    if nbytes == 0:
        return None
    packed = torch.empty(int(nbytes), dtype=torch.uint8, device=t.device)
    _call("cpc_conv_pack %s" % ("x" if operand == 0 else "dy"), 0.0, lib.cpc_conv_pack, _ptr(t), _ptr(packed), ctypes.byref(p),
          operand, _stream(), nbytes=4.0 * t.numel() + float(nbytes))
    return packed


class _ConvFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, stride, pad_top, pad_left, out_hw, relu, precision):
        y, saved = _conv_forward(ctx, x, weight, bias, stride, pad_top, pad_left, out_hw, relu, precision)
        ctx.save_for_backward(*saved)
        return y

    @staticmethod
    def backward(ctx, dy):
        return _conv_backward(ctx, ctx.saved_tensors, dy) + (None,) * 6


class _ConvPoolFunction(torch.autograd.Function):
    """(conv2d(x), max_pool2d(x)) as ONE node for an input that feeds both (the first conv and the pooled residual branch
    of a ScalogramEncoderBlock, scalogram_model.py:446-450).  Forward is the two plain kernels; backward lets the conv's
    data gradient write dx and the pooling add its share in place (cpc_maxpool_bwd_accumulate) instead of a zero-filled
    pooling gradient plus autograd's add pass over the block input."""

    @staticmethod
    def forward(ctx, x, weight, bias, stride, pad_top, pad_left, out_hw, relu, precision, kernel, ceil_mode):
        y, saved = _conv_forward(ctx, x, weight, bias, stride, pad_top, pad_left, out_hw, relu, precision)
        lib = _lib.load()
        x = saved[0]
        p = _pool_params(tuple(x.shape), kernel, ceil_mode)
        if p.h_out <= 0 or p.w_out <= 0:
            raise ValueError("max_pool2d output would be empty for input %s, kernel %d" % (tuple(x.shape), kernel))
        pooled = torch.empty((p.batch, p.channels, p.h_out, p.w_out), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            _call("cpc_maxpool_fwd b%d %dx%dx%d k%d" % (p.batch, p.channels, p.h_in, p.w_in, kernel), 0.0,
                  lib.cpc_maxpool_fwd, _ptr(x), _ptr(pooled), ctypes.byref(p), _stream(),
                  nbytes=4.0 * (x.numel() + pooled.numel()))
        ctx.pool = (kernel, ceil_mode)
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(*saved)
        return y, pooled

    @staticmethod
    @once_differentiable
    def backward(ctx, dy, d_pooled):
        saved = ctx.saved_tensors
        x = saved[0]
        kernel, ceil_mode = ctx.pool
        lib = _lib.load()
        dx = dw = db = None
        if dy is not None:
            dx, dw, db = _conv_backward(ctx, saved, dy)
        if d_pooled is not None and ctx.needs_input_grad[0]:
            p = _pool_params(tuple(x.shape), kernel, ceil_mode)
            d_pooled = d_pooled.contiguous()
            with torch.cuda.device(x.device):
                if dx is None:
                    dx = torch.empty_like(x)
                    _call("cpc_maxpool_bwd b%d %dx%dx%d k%d" % (p.batch, p.channels, p.h_in, p.w_in, kernel), 0.0,
                          lib.cpc_maxpool_bwd, _ptr(x), _ptr(d_pooled), _ptr(dx), ctypes.byref(p), _stream(),
                          nbytes=4.0 * (2 * x.numel() + d_pooled.numel()))
                else:
                    _call("cpc_maxpool_bwd b%d %dx%dx%d k%d +=" % (p.batch, p.channels, p.h_in, p.w_in, kernel), 0.0,
                          lib.cpc_maxpool_bwd_accumulate, _ptr(x), _ptr(d_pooled), _ptr(dx), ctypes.byref(p), _stream(),
                          nbytes=4.0 * (3 * x.numel() + d_pooled.numel()))
        return (dx, dw, db) + (None,) * 8


def _conv_forward(ctx, x, weight, bias, stride, pad_top, pad_left, out_hw, relu, precision):
    """Body of the conv nodes' forward: returns y and the tensors to save."""
    _require_cuda(x, weight, bias)
    lib = _lib.load()
    x = x.contiguous()
    w = weight.contiguous()
    if x.dtype != torch.float32 or w.dtype != torch.float32:
        raise _lib.CpcError("conv expects fp32 tensors (precision is a kernel-internal setting)")
    p = _conv_params(tuple(x.shape), tuple(w.shape), stride, pad_top, pad_left, out_hw, relu, precision)
    y = torch.empty((x.shape[0], w.shape[0], out_hw[0], out_hw[1]), dtype=torch.float32, device=x.device)
    ws = _workspace(lib.cpc_conv_workspace_bytes(ctypes.byref(p), 0), x.device)
    with torch.cuda.device(x.device):
        # the packed copy of x serves the forward pass now and the weight gradient later
        keep = ctx.needs_input_grad[1]                      # (torch.is_grad_enabled() is always False in here)
        packed_x = _pack_operand(lib, x, p, 0) if keep else None
        _call(_conv_key("cpc_conv_fwd", p), _conv_flops(p), lib.cpc_conv_fwd_ex, _ptr(x), _ptr(w),
              _ptr(bias.contiguous() if bias is not None else None), _ptr(y), ctypes.byref(p), _ptr(packed_x),
              _ptr(ws), ws.numel() if ws is not None else 0, _stream())
    ctx.params = (tuple(x.shape), tuple(w.shape), stride, pad_top, pad_left, out_hw, precision)
    ctx.has_bias = bias is not None
    ctx.relu = relu
    return y, (x, w, y if relu else None, packed_x)


def _conv_backward(ctx, saved, dy):
    """Body of the conv nodes' backward: (dx, dw, db)."""
    x, w, y, packed_x = saved
    lib = _lib.load()
    x_shape, w_shape, stride, pad_top, pad_left, out_hw, precision = ctx.params
    if ctx.relu:
        # gradient of the fused ReLU epilogue: one pass (aten's relu backward) outside second-order mode, the plainly
        # differentiable expression under create_graph
        dy = dy * (y > 0).to(dy.dtype) if torch.is_grad_enabled() else torch.ops.aten.threshold_backward(dy, y, 0.0)
    dy = dy.contiguous()
    if torch.is_grad_enabled():
        # backward under create_graph=True: record dgrad / wgrad as differentiable nodes
        geom = (x_shape, w_shape, stride, pad_top, pad_left, out_hw, precision)
        dx = _ConvDgradFunction.apply(dy, w, geom) if ctx.needs_input_grad[0] else None
        dw = _ConvWgradFunction.apply(x, dy, geom) if ctx.needs_input_grad[1] else None
        db = dy.sum(dim=(0, 2, 3)) if (ctx.has_bias and ctx.needs_input_grad[2]) else None
        return dx, dw, db
    p = _conv_params(x_shape, w_shape, stride, pad_top, pad_left, out_hw, False, precision)
    dx = dw = db = None
    need_dx = ctx.needs_input_grad[0]
    need_dw = ctx.needs_input_grad[1] or (ctx.has_bias and ctx.needs_input_grad[2])
    with torch.cuda.device(dy.device):
        packed_dy = None
        if need_dw:
            nbytes = lib.cpc_conv_packed_bytes(ctypes.byref(p), 1)
            if nbytes and ctx.has_bias:
                # the packing pass over dy also reduces the bias gradient (dy is read once for both)
                packed_dy = torch.empty(int(nbytes), dtype=torch.uint8, device=dy.device)
                db = torch.empty(w_shape[0], dtype=torch.float32, device=dy.device)
                _call("cpc_conv_pack dy", 0.0, lib.cpc_conv_pack_dy, _ptr(dy), _ptr(packed_dy), _ptr(db), ctypes.byref(p),
                      _stream(), nbytes=4.0 * dy.numel() + float(nbytes))
            else:
                packed_dy = _pack_operand(lib, dy, p, 1)
        # data and weight gradient are independent: when both are small (neither fills the 148 SMs for long) the weight
        # gradient runs on a side stream next to the data gradient (fork / join inside this call, so every buffer
        # the side stream touches outlives the join; under graph capture the fork becomes a parallel branch)
        side = None
        if need_dx and need_dw and _profiler is None and _conv_flops(p) < _OVERLAP_MAX_FLOPS and not _switch("CPC_NO_BWD_OVERLAP"):
            side = _side_stream(dy.device)
            side.wait_stream(torch.cuda.current_stream(dy.device))
        ws_d = ws_w = None
        if need_dx:
            dx = torch.empty(x_shape, dtype=torch.float32, device=dy.device)
            ws_d = _workspace(lib.cpc_conv_workspace_bytes(ctypes.byref(p), 1), dy.device)
            _call(_conv_key("cpc_conv_dgrad", p), _conv_flops(p), lib.cpc_conv_dgrad_ex, _ptr(dy), _ptr(w), _ptr(dx),
                  ctypes.byref(p), _ptr(packed_dy), _ptr(ws_d), ws_d.numel() if ws_d is not None else 0, _stream())
        if need_dw:
            dw = torch.empty(w_shape, dtype=torch.float32, device=dy.device)
            db_here = None                                   # bias gradient still to be computed by the wgrad call
            if ctx.has_bias and db is None:
                db = db_here = torch.empty(w_shape[0], dtype=torch.float32, device=dy.device)
            ws_w = _workspace(lib.cpc_conv_workspace_bytes(ctypes.byref(p), 2), dy.device)
            with (torch.cuda.stream(side) if side is not None else contextlib.nullcontext()):
                _call(_conv_key("cpc_conv_wgrad", p), _conv_flops(p), lib.cpc_conv_wgrad_ex, _ptr(x), _ptr(dy), _ptr(dw),
                      _ptr(db_here), ctypes.byref(p), _ptr(packed_x), _ptr(packed_dy), _ptr(ws_w),
                      ws_w.numel() if ws_w is not None else 0, _stream())
        if side is not None:
            torch.cuda.current_stream(dy.device).wait_stream(side)
    return dx, dw, db


class _ConvDgradFunction(torch.autograd.Function):
    """dx = conv_transpose(dy, w) as a differentiable node (bilinear in dy and w):
    d/d(dy) = conv_fwd(g, w),  d/d(w) = wgrad(x := g, dy)."""

    @staticmethod
    def forward(ctx, dy, w, geom):
        _require_cuda(dy, w)
        lib = _lib.load()
        x_shape, w_shape, stride, pad_top, pad_left, out_hw, precision = geom
        dy, w = dy.contiguous(), w.contiguous()
        p = _conv_params(x_shape, w_shape, stride, pad_top, pad_left, out_hw, False, precision)
        dx = torch.empty(x_shape, dtype=torch.float32, device=dy.device)
        ws = _workspace(lib.cpc_conv_workspace_bytes(ctypes.byref(p), 1), dy.device)
        with torch.cuda.device(dy.device):
            _call(_conv_key("cpc_conv_dgrad", p), _conv_flops(p), lib.cpc_conv_dgrad_ex, _ptr(dy), _ptr(w), _ptr(dx),
                  ctypes.byref(p), _ptr(None), _ptr(ws), ws.numel() if ws is not None else 0, _stream())
        ctx.geom = geom
        ctx.save_for_backward(dy, w)
        return dx

    @staticmethod
    def backward(ctx, g):
        dy, w = ctx.saved_tensors
        x_shape, w_shape, stride, pad_top, pad_left, out_hw, precision = ctx.geom
        g = g.contiguous()
        g_dy = (_ConvFunction.apply(g, w, None, stride, pad_top, pad_left, out_hw, False, precision)
                if ctx.needs_input_grad[0] else None)
        g_w = _ConvWgradFunction.apply(g, dy, ctx.geom) if ctx.needs_input_grad[1] else None
        return g_dy, g_w, None


class _ConvWgradFunction(torch.autograd.Function):
    """dw = wgrad(x, dy) as a differentiable node (bilinear in x and dy):
    d/d(x) = conv_transpose(dy, g),  d/d(dy) = conv_fwd(x, g)."""

    @staticmethod
    def forward(ctx, x, dy, geom):
        _require_cuda(x, dy)
        lib = _lib.load()
        x_shape, w_shape, stride, pad_top, pad_left, out_hw, precision = geom
        x, dy = x.contiguous(), dy.contiguous()
        p = _conv_params(x_shape, w_shape, stride, pad_top, pad_left, out_hw, False, precision)
        dw = torch.empty(w_shape, dtype=torch.float32, device=dy.device)
        ws = _workspace(lib.cpc_conv_workspace_bytes(ctypes.byref(p), 2), dy.device)
        with torch.cuda.device(dy.device):
            _call(_conv_key("cpc_conv_wgrad", p), _conv_flops(p), lib.cpc_conv_wgrad_ex, _ptr(x), _ptr(dy), _ptr(dw),
                  _ptr(None), ctypes.byref(p), _ptr(None), _ptr(None), _ptr(ws), ws.numel() if ws is not None else 0,
                  _stream())
        ctx.geom = geom
        ctx.save_for_backward(x, dy)
        return dw

    @staticmethod
    def backward(ctx, g):
        x, dy = ctx.saved_tensors
        x_shape, w_shape, stride, pad_top, pad_left, out_hw, precision = ctx.geom
        g = g.contiguous()
        g_x = _ConvDgradFunction.apply(dy, g, ctx.geom) if ctx.needs_input_grad[0] else None
        g_dy = (_ConvFunction.apply(x, g, None, stride, pad_top, pad_left, out_hw, False, precision)
                if ctx.needs_input_grad[1] else None)
        return g_x, g_dy, None


def conv2d(x, weight, bias=None, stride=(1, 1), padding=(0, 0), extra_top=0, relu=False, precision=None):
    """y = [relu](conv2d(zero_pad_top(x, extra_top), weight, bias, stride, padding)); NCHW fp32.
    Semantics of F.conv2d preceded by nn.ZeroPad2d((0, 0, extra_top, 0)) (scalogram_model.py:389-397)."""
    if isinstance(stride, int):
        stride = (stride, stride)
    if isinstance(padding, int):
        padding = (padding, padding)
    b, c, h, w_in = x.shape
    co, ci, kh, kw = weight.shape
    if ci != c:
        raise ValueError("channel mismatch: input has %d channels, weight expects %d" % (c, ci))
    oh = (h + extra_top + 2 * padding[0] - kh) // stride[0] + 1
    ow = (w_in + 2 * padding[1] - kw) // stride[1] + 1
    if oh <= 0 or ow <= 0:
        raise ValueError("conv output would be empty: input %s kernel %s" % (tuple(x.shape), (kh, kw)))
    return _ConvFunction.apply(x, weight, bias, tuple(stride), extra_top + padding[0], padding[1], (oh, ow), relu,
                               precision or _default_precision)


def conv2d_with_pool(x, weight, bias, stride, padding, extra_top, pool_kernel, pool_ceil_mode, precision=None):
    """``(conv2d(x, ...), max_pool2d(x, pool_kernel, ceil_mode))`` for an input both operators read; same values as the
    two separate calls, one autograd node whose backward needs no add pass over ``x`` (see _ConvPoolFunction)."""
    if isinstance(stride, int):
        stride = (stride, stride)
    if isinstance(padding, int):
        padding = (padding, padding)
    b, c, h, w_in = x.shape
    co, ci, kh, kw = weight.shape
    if ci != c:
        raise ValueError("channel mismatch: input has %d channels, weight expects %d" % (c, ci))
    oh = (h + extra_top + 2 * padding[0] - kh) // stride[0] + 1
    ow = (w_in + 2 * padding[1] - kw) // stride[1] + 1
    if oh <= 0 or ow <= 0:
        raise ValueError("conv output would be empty: input %s kernel %s" % (tuple(x.shape), (kh, kw)))
    return _ConvPoolFunction.apply(x, weight, bias, tuple(stride), extra_top + padding[0], padding[1], (oh, ow), False,
                                   precision or _default_precision, int(pool_kernel), bool(pool_ceil_mode))


def conv1d(x, weight, bias=None, stride=1, padding=0, relu=False, precision=None):
    """F.conv1d semantics (audio_model.py:30-44) through the same kernel family (h = 1)."""
    y = conv2d(x.unsqueeze(2), weight.unsqueeze(2), bias, (1, stride), (0, padding), 0, relu, precision)
    return y.squeeze(2)


def conv_transpose1d(x, weight, stride=1, padding=0, precision=None):
    """F.conv_transpose1d(x, weight, stride=stride, padding=padding) (no bias, no output padding): x (N, C_in, T),
    weight (C_in, C_out, K) -> (N, C_out, (T-1)*stride - 2*padding + K).  It IS the data gradient of the conv1d
    with that weight, so it runs on the dgrad kernels (InverseCQT, constant_q_transform.py:233-236)."""
    n, c_in, t = x.shape
    if weight.shape[0] != c_in:
        raise ValueError("channel mismatch: input has %d channels, weight expects %d" % (c_in, weight.shape[0]))
    c_out, k = weight.shape[1], weight.shape[2]
    length = (t - 1) * stride - 2 * padding + k
    if length <= 0:
        raise ValueError("conv_transpose1d output would be empty")
    geom = ((n, c_out, 1, length), (c_in, c_out, 1, k), (1, stride), 0, padding, (1, t), precision or _default_precision)
    return _ConvDgradFunction.apply(x.unsqueeze(2), weight.unsqueeze(2), geom).squeeze(2)


# --------------------------------------------------------------------------------------------------
# depthwise convolution (the first half of Conv2dSeparable)
# --------------------------------------------------------------------------------------------------

class _DepthwiseConvFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, stride, pad_top, pad_left, out_hw):
        _require_cuda(x, weight)
        lib = _lib.load()
        x, w = x.contiguous(), weight.contiguous()
        if x.dtype != torch.float32 or w.dtype != torch.float32:
            raise _lib.CpcError("depthwise conv expects fp32 tensors")
        c = x.shape[1]
        p = _conv_params(tuple(x.shape), (c, c, w.shape[2], w.shape[3]), stride, pad_top, pad_left, out_hw, False, "fp32")
        y = torch.empty((x.shape[0], c, out_hw[0], out_hw[1]), dtype=torch.float32, device=x.device)
        taps = w.shape[2] * w.shape[3]
        with torch.cuda.device(x.device):
            _call("cpc_dwconv_fwd b%d %dx%dx%d k%dx%d" % (x.shape[0], c, x.shape[2], x.shape[3], w.shape[2], w.shape[3]),
                  2.0 * taps * y.numel(), lib.cpc_dwconv_fwd, _ptr(x), _ptr(w), _ptr(y), ctypes.byref(p), _stream(),
                  nbytes=4.0 * (x.numel() + y.numel()))
        ctx.geom = (tuple(x.shape), tuple(w.shape), stride, pad_top, pad_left, out_hw)
        ctx.save_for_backward(x, w)
        return y

    @staticmethod
    @once_differentiable                                         # second-order mode uses F.conv2d(groups=C) instead
    def backward(ctx, dy):
        x, w = ctx.saved_tensors
        lib = _lib.load()
        x_shape, w_shape, stride, pad_top, pad_left, out_hw = ctx.geom
        c = x_shape[1]
        p = _conv_params(x_shape, (c, c, w_shape[2], w_shape[3]), stride, pad_top, pad_left, out_hw, False, "fp32")
        dy = dy.contiguous()
        dx = dw = None
        tag = "b%d %dx%dx%d k%dx%d" % (x_shape[0], c, x_shape[2], x_shape[3], w_shape[2], w_shape[3])
        with torch.cuda.device(dy.device):
            if ctx.needs_input_grad[0]:
                dx = torch.empty(x_shape, dtype=torch.float32, device=dy.device)
                _call("cpc_dwconv_dgrad " + tag, 0.0, lib.cpc_dwconv_dgrad, _ptr(dy), _ptr(w), _ptr(dx), ctypes.byref(p),
                      _stream(), nbytes=4.0 * (dx.numel() + dy.numel()))
            if ctx.needs_input_grad[1]:
                dw = torch.empty(w_shape, dtype=torch.float32, device=dy.device)
                _call("cpc_dwconv_wgrad " + tag, 0.0, lib.cpc_dwconv_wgrad, _ptr(x), _ptr(dy), _ptr(dw), ctypes.byref(p),
                      _stream(), nbytes=4.0 * (x.numel() + dy.numel()))
        return dx, dw, None, None, None, None


def depthwise_conv2d(x, weight, stride=(1, 1), padding=(0, 0), extra_top=0):
    """F.conv2d(zero_pad_top(x, extra_top), weight, None, stride, padding, groups=C) for weight (C, 1, kh, kw)."""
    if isinstance(stride, int):
        stride = (stride, stride)
    if isinstance(padding, int):
        padding = (padding, padding)
    b, c, h, w_in = x.shape
    if weight.shape[0] != c or weight.shape[1] != 1:
        raise ValueError("depthwise weight must be (C, 1, kh, kw) with C = %d, got %s" % (c, tuple(weight.shape)))
    kh, kw = weight.shape[2], weight.shape[3]
    oh = (h + extra_top + 2 * padding[0] - kh) // stride[0] + 1
    ow = (w_in + 2 * padding[1] - kw) // stride[1] + 1
    if oh <= 0 or ow <= 0:
        raise ValueError("conv output would be empty: input %s kernel %s" % (tuple(x.shape), (kh, kw)))
    if _second_order:
        import torch.nn.functional as F
        return F.conv2d(F.pad(x, (0, 0, extra_top, 0)) if extra_top else x, weight, None, stride, padding, groups=c)
    return _DepthwiseConvFunction.apply(x, weight, tuple(stride), extra_top + padding[0], padding[1], (oh, ow))


# --------------------------------------------------------------------------------------------------
# fused BatchNorm2d + ReLU (+ cropped residual add + ReLU)
# --------------------------------------------------------------------------------------------------

def _bn_params(x_shape, res_shape, res_off, relu, outer_relu, training, eps, momentum, packed_planes=0):
    p = _lib.BnParams()
    p.packed_planes = int(packed_planes)                         # *_packed calls: 1 = hi plane only (bf16 conv mode)
    p.batch, p.channels, p.height, p.width = x_shape
    if res_shape is not None:
        p.res_height, p.res_width = res_shape[2], res_shape[3]
        p.res_off_h, p.res_off_w = res_off
    p.relu, p.outer_relu, p.training = int(relu), int(outer_relu), int(training)
    p.eps, p.momentum = float(eps), float(momentum)
    return p


def _bn_mask(lib, p, device):
    """Bit-mask buffer for the ReLU behind the residual add of (p), or None when the shape has none (or the switch
    CPC_NO_BN_MASK asks for the recomputing kernels)."""
    if _switch("CPC_NO_BN_MASK"):
        return None
    n = int(lib.cpc_bn_mask_bytes(ctypes.byref(p)))
    return torch.empty(n, dtype=torch.uint8, device=device) if n else None


def _bn_key(tag, p):
    return "%s b%d %dx%dx%d%s" % (tag, p.batch, p.channels, p.height, p.width, " +res" if p.res_height else "")


class _BnReluFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, gamma, beta, running_mean, running_var, residual, res_off, relu, outer_relu, training, eps,
                momentum):
        _require_cuda(x, gamma, beta, running_mean, running_var, residual)
        lib = _lib.load()
        x = x.contiguous()
        if residual is not None:
            residual = residual.contiguous()
            if residual.shape[:2] != x.shape[:2]:
                raise ValueError("residual %s does not match %s" % (tuple(residual.shape), tuple(x.shape)))
        if x.dtype != torch.float32 or x.dim() != 4:
            raise _lib.CpcError("bn_relu expects a 4-d fp32 tensor")
        p = _bn_params(tuple(x.shape), None if residual is None else tuple(residual.shape), res_off, relu, outer_relu,
                       training, eps, momentum)
        c = x.shape[1]
        out = torch.empty_like(x)
        save_mean = torch.empty(c, dtype=torch.float32, device=x.device)
        save_rstd = torch.empty(c, dtype=torch.float32, device=x.device)
        ws = _workspace(lib.cpc_bn_relu_workspace_bytes(ctypes.byref(p)), x.device)
        n = x.numel()
        mask = _bn_mask(lib, p, x.device) if any(ctx.needs_input_grad) else None
        with torch.cuda.device(x.device):
            _call(_bn_key("cpc_bn_relu_fwd", p), 0.0, lib.cpc_bn_relu_fwd_mask, _ptr(x), _ptr(gamma), _ptr(beta),
                  _ptr(running_mean), _ptr(running_var), _ptr(residual), _ptr(out), _ptr(save_mean), _ptr(save_rstd),
                  _ptr(mask), ctypes.byref(p), _ptr(ws), ws.numel(), _stream(),
                  nbytes=4.0 * n * ((3 if training else 2) + (1 if residual is not None else 0)))
        ctx.cfg = (tuple(x.shape), None if residual is None else tuple(residual.shape), res_off, relu, outer_relu,
                   training, eps, momentum)
        ctx.has_residual = residual is not None
        # with the saved mask the residual's values are not needed again: keep only what autograd must return
        ctx.save_for_backward(x, gamma, beta, save_mean, save_rstd, residual if mask is None else None, mask)
        return out

    @staticmethod
    @once_differentiable                                         # second-order mode uses the literal modules instead
    def backward(ctx, dout):
        x, gamma, beta, save_mean, save_rstd, residual, mask = ctx.saved_tensors
        lib = _lib.load()
        x_shape, res_shape, res_off, relu, outer_relu, training, eps, momentum = ctx.cfg
        p = _bn_params(x_shape, res_shape, res_off, relu, outer_relu, training, eps, momentum)
        dout = dout.contiguous()
        dx = torch.empty_like(x)
        dgamma = torch.empty_like(gamma) if gamma is not None else None
        dbeta = torch.empty_like(beta) if beta is not None else None
        d_res = (torch.empty(res_shape, dtype=torch.float32, device=x.device)
                 if (ctx.has_residual and ctx.needs_input_grad[5]) else None)
        ws = _workspace(lib.cpc_bn_relu_workspace_bytes(ctypes.byref(p)), x.device)
        n = x.numel()
        # the residual pointer only says "there is a residual" when the mask is given; x stands in for it
        res_arg = residual if residual is not None else (x if ctx.has_residual else None)
        with torch.cuda.device(x.device):
            _call(_bn_key("cpc_bn_relu_bwd", p), 0.0, lib.cpc_bn_relu_bwd_mask, _ptr(dout), _ptr(x), _ptr(gamma),
                  _ptr(beta), _ptr(save_mean), _ptr(save_rstd), _ptr(res_arg), _ptr(mask), _ptr(dx), _ptr(dgamma),
                  _ptr(dbeta), _ptr(d_res), ctypes.byref(p), _ptr(ws), ws.numel(), _stream(),
                  nbytes=4.0 * n * (5 + (2 if (residual is not None and outer_relu) else 0) + (1 if d_res is not None else 0))
                  + (2.0 * mask.numel() if mask is not None else 0.0))
        return dx, dgamma, dbeta, None, None, d_res, None, None, None, None, None, None


def bn_relu(x, bn, residual=None, res_off=(0, 0), relu=True, outer_relu=False):
    """``relu_if(outer_relu, relu_if(relu, bn(x)) + crop(residual))`` for an ``nn.BatchNorm2d`` module ``bn``
    (train mode: batch statistics + running-stat update; eval mode: running statistics).  One fused kernel family
    forward, one backward (scalogram_model.py:399-431, 451-472, 523-527)."""
    training = bn.training or bn.running_mean is None
    momentum = bn.momentum
    if training and bn.track_running_stats and bn.num_batches_tracked is not None:
        bn.num_batches_tracked.add_(1)
        if momentum is None:
            momentum = 1.0 / float(bn.num_batches_tracked)
    if momentum is None:
        momentum = 0.0
    rm = bn.running_mean if bn.track_running_stats else None
    rv = bn.running_var if bn.track_running_stats else None
    return _BnReluFunction.apply(x, bn.weight, bn.bias, rm, rv, residual, tuple(res_off), bool(relu), bool(outer_relu),
                                 bool(training), bn.eps, momentum)


def _bn_state(bn):
    """(training, momentum, running_mean, running_var) of an nn.BatchNorm2d for one forward call, advancing
    num_batches_tracked like nn.BatchNorm2d.forward does."""
    training = bn.training or bn.running_mean is None
    momentum = bn.momentum
    if training and bn.track_running_stats and bn.num_batches_tracked is not None:
        bn.num_batches_tracked.add_(1)
        if momentum is None:
            momentum = 1.0 / float(bn.num_batches_tracked)
    if momentum is None:
        momentum = 0.0
    rm = bn.running_mean if bn.track_running_stats else None
    rv = bn.running_var if bn.track_running_stats else None
    return bool(training), momentum, rm, rv


class _BlockTailFunction(torch.autograd.Function):
    """Everything of a ScalogramEncoderBlock behind its first conv as ONE autograd node (scalogram_model.py:399-431,
    451-472):   out = relu_if(outer, relu(bn1(conv_b(relu(bn0(y_a))))) + crop(residual)).

    Inside the node the activation between bn0 and conv_b and the gradient between bn1 and conv_b exist only as the
    bf16 hi/lo operand planes the row-streaming conv kernels read: bn0 writes them instead of an fp32 tensor, bn1's
    backward writes dy the same way (plus its per-channel sum = conv_b's bias gradient).  Two fp32 tensors, two packing
    passes and the bias-gradient pass of the unfused chain disappear; every value is computed by the same kernels."""

    @staticmethod
    def forward(ctx, y_a, g0, b0, rm0, rv0, w, bias, g1, b1, rm1, rv1, residual, cfg):
        (top, out_hw, res_off, outer_relu, tr0, eps0, mom0, tr1, eps1, mom1, precision) = cfg
        _require_cuda(y_a, w, residual)
        lib = _lib.load()
        y_a = y_a.contiguous()
        w = w.contiguous()
        if residual is not None:
            residual = residual.contiguous()
        dev = y_a.device
        B, C, H, W = y_a.shape
        # bn0 + relu -> packed h
        planes = 1 if precision == "bf16" else 2                 # operand planes the conv kernels of this mode read
        p0 = _bn_params((B, C, H, W), None, (0, 0), True, False, tr0, eps0, mom0, planes)
        packed_h = torch.empty(int(lib.cpc_bn_packed_bytes(ctypes.byref(p0))), dtype=torch.uint8, device=dev)
        mean0 = torch.empty(C, dtype=torch.float32, device=dev)
        rstd0 = torch.empty(C, dtype=torch.float32, device=dev)
        ws = _workspace(lib.cpc_bn_relu_workspace_bytes(ctypes.byref(p0)), dev)
        pc = _conv_params((B, C, H, W), tuple(w.shape), (1, 1), top, 0, out_hw, False, precision)
        co = w.shape[0]
        y_b = torch.empty((B, co, out_hw[0], out_hw[1]), dtype=torch.float32, device=dev)
        p1 = _bn_params(tuple(y_b.shape), None if residual is None else tuple(residual.shape), res_off, True, outer_relu,
                        tr1, eps1, mom1)
        out = torch.empty_like(y_b)
        mean1 = torch.empty(co, dtype=torch.float32, device=dev)
        rstd1 = torch.empty(co, dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _call(_bn_key("cpc_bn_relu_fwd", p0) + " ->packed", 0.0, lib.cpc_bn_relu_fwd_packed, _ptr(y_a), _ptr(g0), _ptr(b0),
                  _ptr(rm0), _ptr(rv0), _ptr(None), _ptr(packed_h), _ptr(mean0), _ptr(rstd0), ctypes.byref(p0), _ptr(ws),
                  ws.numel(), _stream(), nbytes=4.0 * y_a.numel() * (2 if tr0 else 1) + float(packed_h.numel()))
            wsc = _workspace(lib.cpc_conv_workspace_bytes(ctypes.byref(pc), 0), dev)
            _call(_conv_key("cpc_conv_fwd", pc), _conv_flops(pc), lib.cpc_conv_fwd_ex, _ptr(None), _ptr(w),
                  _ptr(bias.contiguous() if bias is not None else None), _ptr(y_b), ctypes.byref(pc), _ptr(packed_h),
                  _ptr(wsc), wsc.numel() if wsc is not None else 0, _stream())
            ws1 = _workspace(lib.cpc_bn_relu_workspace_bytes(ctypes.byref(p1)), dev)
            n1 = y_b.numel()
            mask = _bn_mask(lib, p1, dev) if any(ctx.needs_input_grad) else None
            _call(_bn_key("cpc_bn_relu_fwd", p1), 0.0, lib.cpc_bn_relu_fwd_mask, _ptr(y_b), _ptr(g1), _ptr(b1), _ptr(rm1),
                  _ptr(rv1), _ptr(residual), _ptr(out), _ptr(mean1), _ptr(rstd1), _ptr(mask), ctypes.byref(p1), _ptr(ws1),
                  ws1.numel(), _stream(), nbytes=4.0 * n1 * ((3 if tr1 else 2) + (1 if residual is not None else 0)))
        ctx.cfg = cfg
        ctx.has_bias = bias is not None
        ctx.res_shape = None if residual is None else tuple(residual.shape)
        ctx.save_for_backward(y_a, g0, b0, mean0, rstd0, packed_h, w, y_b, g1, b1, mean1, rstd1,
                              residual if mask is None else None, mask)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, dout):
        y_a, g0, b0, mean0, rstd0, packed_h, w, y_b, g1, b1, mean1, rstd1, residual, mask = ctx.saved_tensors
        (top, out_hw, res_off, outer_relu, tr0, eps0, mom0, tr1, eps1, mom1, precision) = ctx.cfg
        lib = _lib.load()
        dev = dout.device
        dout = dout.contiguous()
        B, C, H, W = y_a.shape
        co = w.shape[0]
        planes = 1 if precision == "bf16" else 2
        p1 = _bn_params(tuple(y_b.shape), ctx.res_shape, res_off, True, outer_relu, tr1, eps1, mom1, planes)
        # with the saved mask the residual is not read: y_b stands in for "there is a residual"
        res_arg = residual if residual is not None else (y_b if ctx.res_shape is not None else None)
        pc = _conv_params((B, C, H, W), tuple(w.shape), (1, 1), top, 0, out_hw, False, precision)
        p0 = _bn_params((B, C, H, W), None, (0, 0), True, False, tr0, eps0, mom0)
        packed_dy = torch.empty(int(lib.cpc_bn_packed_bytes(ctypes.byref(p1))), dtype=torch.uint8, device=dev)
        db = torch.empty(co, dtype=torch.float32, device=dev) if ctx.has_bias else None
        dg1 = torch.empty_like(g1) if g1 is not None else None
        dbt1 = torch.empty_like(b1) if b1 is not None else None
        d_res = (torch.empty(ctx.res_shape, dtype=torch.float32, device=dev)
                 if (ctx.res_shape is not None and ctx.needs_input_grad[11]) else None)
        dh = torch.empty((B, C, H, W), dtype=torch.float32, device=dev)
        dw = torch.empty_like(w)
        dy_a = torch.empty_like(y_a)
        dg0 = torch.empty_like(g0) if g0 is not None else None
        dbt0 = torch.empty_like(b0) if b0 is not None else None
        with torch.cuda.device(dev):
            ws1 = _workspace(lib.cpc_bn_relu_workspace_bytes(ctypes.byref(p1)), dev)
            n1 = y_b.numel()
            _call(_bn_key("cpc_bn_relu_bwd", p1) + " ->packed", 0.0, lib.cpc_bn_relu_bwd_packed_mask, _ptr(dout), _ptr(y_b),
                  _ptr(g1), _ptr(b1), _ptr(mean1), _ptr(rstd1), _ptr(res_arg), _ptr(mask), _ptr(packed_dy), _ptr(db),
                  _ptr(dg1), _ptr(dbt1), _ptr(d_res), ctypes.byref(p1), _ptr(ws1), ws1.numel(), _stream(),
                  nbytes=4.0 * n1 * (5 + (2 if (residual is not None and outer_relu) else 0) + (1 if d_res is not None else 0))
                  + (2.0 * mask.numel() if mask is not None else 0.0))
            wsd = _workspace(lib.cpc_conv_workspace_bytes(ctypes.byref(pc), 1), dev)
            _call(_conv_key("cpc_conv_dgrad", pc), _conv_flops(pc), lib.cpc_conv_dgrad_ex, _ptr(None), _ptr(w), _ptr(dh),
                  ctypes.byref(pc), _ptr(packed_dy), _ptr(wsd), wsd.numel() if wsd is not None else 0, _stream())
            wsw = _workspace(lib.cpc_conv_workspace_bytes(ctypes.byref(pc), 2), dev)
            _call(_conv_key("cpc_conv_wgrad", pc), _conv_flops(pc), lib.cpc_conv_wgrad_ex, _ptr(None), _ptr(None), _ptr(dw),
                  _ptr(None), ctypes.byref(pc), _ptr(packed_h), _ptr(packed_dy), _ptr(wsw),
                  wsw.numel() if wsw is not None else 0, _stream())
            ws0 = _workspace(lib.cpc_bn_relu_workspace_bytes(ctypes.byref(p0)), dev)
            _call(_bn_key("cpc_bn_relu_bwd", p0), 0.0, lib.cpc_bn_relu_bwd, _ptr(dh), _ptr(y_a), _ptr(g0), _ptr(b0), _ptr(mean0),
                  _ptr(rstd0), _ptr(None), _ptr(dy_a), _ptr(dg0), _ptr(dbt0), _ptr(None), ctypes.byref(p0), _ptr(ws0),
                  ws0.numel(), _stream(), nbytes=4.0 * y_a.numel() * 5)
        return dy_a, dg0, dbt0, None, None, dw, db, dg1, dbt1, None, None, d_res, None


def block_tail_eligible(y_a, bn0, conv, top, bn1):
    """True when ``relu(bn0(y_a)) -> conv -> bn1`` can run as one node with packed intermediates: kh x 1 stride-1 conv
    without horizontal padding on the row-streaming kernels (forward, data and weight gradient), fp32-faithful mode,
    affine batch norms, first-order autograd.  Both operand modes: fp32-faithful (hi + lo planes) and bf16 (hi plane)."""
    if _switch("CPC_NO_BLOCK_TAIL") or _second_order:
        return False
    if not (y_a.is_cuda and y_a.dtype == torch.float32 and y_a.dim() == 4 and y_a.shape[3] % 2 == 0):
        return False                                             # the packed-output kernels own pairs of columns
    w = conv.weight
    if (tuple(conv.stride) != (1, 1) or w.shape[3] != 1 or conv.padding[1] != 0 or conv.groups != 1
            or tuple(conv.dilation) != (1, 1) or w.shape[1] != y_a.shape[1]):
        return False
    for bn in (bn0, bn1):
        if bn.weight is None or bn.bias is None:
            return False
    B, C, H, W = y_a.shape
    oh = H + top + 2 * conv.padding[0] - w.shape[2] + 1
    if oh <= 0:
        return False
    p = _conv_params((B, C, H, W), tuple(w.shape), (1, 1), top + conv.padding[0], 0, (oh, W), False, _default_precision)
    lib = _lib.load()
    return all(lib.cpc_conv_kernel_family(ctypes.byref(p), which) in (2, 3) for which in (0, 1, 2))


def block_tail(y_a, bn0, conv, top, bn1, residual=None, res_off=(0, 0), outer_relu=False):
    """relu_if(outer_relu, relu(bn1(conv(pad_top(relu(bn0(y_a)))))) + crop(residual)); see _BlockTailFunction."""
    tr0, mom0, rm0, rv0 = _bn_state(bn0)
    tr1, mom1, rm1, rv1 = _bn_state(bn1)
    w = conv.weight
    pad_top = top + conv.padding[0]
    oh = y_a.shape[2] + top + 2 * conv.padding[0] - w.shape[2] + 1
    cfg = (pad_top, (oh, y_a.shape[3]), tuple(res_off), bool(outer_relu), tr0, bn0.eps, mom0, tr1, bn1.eps, mom1,
           _default_precision)
    return _BlockTailFunction.apply(y_a, bn0.weight, bn0.bias, rm0, rv0, w, conv.bias, bn1.weight, bn1.bias, rm1, rv1,
                                    residual, cfg)


# --------------------------------------------------------------------------------------------------
# non-overlapping max pooling
# --------------------------------------------------------------------------------------------------

def _pool_params(x_shape, kernel, ceil_mode):
    p = _lib.PoolParams()
    p.batch, p.channels, p.h_in, p.w_in = x_shape
    p.kernel, p.ceil_mode = int(kernel), int(bool(ceil_mode))
    p.h_out = -(-p.h_in // kernel) if ceil_mode else p.h_in // kernel
    p.w_out = -(-p.w_in // kernel) if ceil_mode else p.w_in // kernel
    return p


class _MaxPoolFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, kernel, ceil_mode):
        _require_cuda(x)
        lib = _lib.load()
        x = x.contiguous()
        if x.dtype != torch.float32 or x.dim() != 4:
            raise _lib.CpcError("max_pool2d expects a 4-d fp32 tensor")
        p = _pool_params(tuple(x.shape), kernel, ceil_mode)
        if p.h_out <= 0 or p.w_out <= 0:
            raise ValueError("max_pool2d output would be empty for input %s, kernel %d" % (tuple(x.shape), kernel))
        y = torch.empty((p.batch, p.channels, p.h_out, p.w_out), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            _call("cpc_maxpool_fwd b%d %dx%dx%d k%d" % (p.batch, p.channels, p.h_in, p.w_in, kernel), 0.0,
                  lib.cpc_maxpool_fwd, _ptr(x), _ptr(y), ctypes.byref(p), _stream(), nbytes=4.0 * (x.numel() + y.numel()))
        ctx.cfg = (tuple(x.shape), kernel, ceil_mode)
        ctx.save_for_backward(x)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, dy):
        (x,) = ctx.saved_tensors
        lib = _lib.load()
        x_shape, kernel, ceil_mode = ctx.cfg
        p = _pool_params(x_shape, kernel, ceil_mode)
        dy = dy.contiguous()
        dx = torch.empty_like(x)
        with torch.cuda.device(x.device):
            _call("cpc_maxpool_bwd b%d %dx%dx%d k%d" % (p.batch, p.channels, p.h_in, p.w_in, kernel), 0.0,
                  lib.cpc_maxpool_bwd, _ptr(x), _ptr(dy), _ptr(dx), ctypes.byref(p), _stream(),
                  nbytes=4.0 * (2 * x.numel() + dy.numel()))
        return dx, None, None


def max_pool2d(x, kernel, ceil_mode=False):
    """nn.MaxPool2d(kernel_size=kernel, ceil_mode=ceil_mode) (stride = kernel, no padding) on the B200 kernels."""
    return _MaxPoolFunction.apply(x, int(kernel), bool(ceil_mode))


# --------------------------------------------------------------------------------------------------
# InfoNCE
# --------------------------------------------------------------------------------------------------

def _nce_key(tag, p):
    return "%s b%d k%d e%d %s" % (tag, p.batch, p.steps, p.enc, "all-steps" if p.all_steps else "per-step")


def _nce_pairs_e(p):
    n = p.batch * p.steps
    return float(n * n * p.enc) if p.all_steps else float(p.steps * p.batch * p.batch * p.enc)


def _nce_flops(p):
    """Forward: the score tile, 2 operations per (pair, e) for a dot product, 3 for (p - z)^2 (subtract + fma)."""
    return (3.0 if p.score_kind == _lib.SCORE_DIFFERENCE else 2.0) * _nce_pairs_e(p)


def _nce_bwd_flops(p):
    """Backward: the score tile recomputed, then the two tile products G.Z and G^T.P (2 operations each)."""
    return _nce_flops(p) + 4.0 * _nce_pairs_e(p)


def _nce_params(pred, targets, all_steps, kind, reg, precision):
    p = _lib.InfoNceParams()
    p.batch, p.steps, p.enc = pred.shape
    p.all_steps = int(bool(all_steps))
    p.score_kind = {"linear": _lib.SCORE_LINEAR, "softplus": _lib.SCORE_SOFTPLUS,
                    "difference": _lib.SCORE_DIFFERENCE}[kind]
    p.regularization = float(reg)
    p.tgt_stride_b, p.tgt_stride_e, p.tgt_stride_k = targets.stride()
    p.precision = _PRECISION[precision]
    p.flags = _lib.INFONCE_FLAG_NO_TENSOR if _switch("CPC_NO_TENSOR_INFONCE") else 0
    return p


class _InfoNceFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, targets, all_steps, kind, reg, precision):
        _require_cuda(pred, targets)
        lib = _lib.load()
        if pred.dtype != torch.float32 or targets.dtype != torch.float32:
            raise _lib.CpcError("infonce expects fp32 tensors")
        b, k, e = pred.shape
        if tuple(targets.shape) != (b, e, k):
            raise ValueError("targets must be (B, E, K) = %s, got %s" % ((b, e, k), tuple(targets.shape)))
        pred = pred.contiguous()
        p = _nce_params(pred, targets, all_steps, kind, reg, precision)
        out = torch.empty(_lib.INFONCE_OUT_FLOATS, dtype=torch.float32, device=pred.device)
        lse = torch.empty(b * k, dtype=torch.float32, device=pred.device)
        ws = _workspace(lib.cpc_infonce_workspace_bytes(ctypes.byref(p), 0), pred.device)
        with torch.cuda.device(pred.device):
            _call(_nce_key("cpc_infonce_fwd", p), _nce_flops(p), lib.cpc_infonce_fwd, _ptr(pred), _ptr(targets),
                  _ptr(out), _ptr(lse), ctypes.byref(p), _ptr(ws), ws.numel() if ws is not None else 0, _stream())
        ctx.args = (all_steps, kind, reg, precision)
        ctx.save_for_backward(pred, targets, lse)
        loss, max_score, loss_noreg, mean_score = out[0], out[1], out[2], out[3]
        ctx.mark_non_differentiable(max_score, loss_noreg, mean_score)
        return loss, max_score, loss_noreg, mean_score

    @staticmethod
    @once_differentiable
    def backward(ctx, g_loss, _g1, _g2, _g3):
        pred, targets, lse = ctx.saved_tensors
        lib = _lib.load()
        all_steps, kind, reg, precision = ctx.args
        p = _nce_params(pred, targets, all_steps, kind, reg, precision)
        g = g_loss.reshape(1).to(torch.float32).contiguous()
        d_pred = torch.empty_like(pred)
        d_tgt = torch.empty(targets.shape, dtype=torch.float32, device=pred.device)
        ws = _workspace(lib.cpc_infonce_workspace_bytes(ctypes.byref(p), 1), pred.device)
        with torch.cuda.device(pred.device):
            _call(_nce_key("cpc_infonce_bwd", p), _nce_bwd_flops(p), lib.cpc_infonce_bwd, _ptr(pred), _ptr(targets),
                  _ptr(lse), _ptr(g), _ptr(d_pred), _ptr(d_tgt), ctypes.byref(p), _ptr(ws),
                  ws.numel() if ws is not None else 0, _stream())
        return d_pred, d_tgt, None, None, None, None


def infonce(pred, targets, all_steps, kind="linear", regularization=0.0, precision=None):
    """Fused InfoNCE.  pred (B,K,E), targets (B,E,K) (any strides).  Returns
    (loss, max_score, loss_without_regulariser, mean_score); only ``loss`` is differentiable.
    Replaces contrastive_estimation_training.py:106-122,141,166.

    kind: "linear" (S = p.z), "softplus" (S = softplus(p.z)) or "difference" (S = 1 / |p - z|^2, the reference's
    difference_score_function).  The difference kind always runs on the fp32 CUDA-core kernels with the squared
    differences summed in fp32, so ``precision="bf16"`` gives bit-identical results to fp32 for it; a prediction equal
    to a target gives S = +inf and a NaN loss.  The reference's literal block gives NaN too when that target is the
    prediction's own, and +inf when it is another candidate's (its logsumexp keeps the +inf where the kernel's
    max-shifted sum gives inf - inf); ``train()`` stops before the optimizer step on a NaN loss."""
    return _InfoNceFunction.apply(pred, targets, bool(all_steps), kind, float(regularization),
                                  precision or _default_precision)


def infonce_validate(pred, targets, all_steps, kind="linear", precision=None):
    """Validation metrics of one batch (contrastive_estimation_training.py:224-247) without materialising the
    (B,K,B,K) score tensor: returns (per_step_losses (K), per_step_accuracy (K), mean_score ()).  The per-step
    losses reproduce the reference's re-viewed ("scrambled") noise term in per-step mode (SURVEY.md Appendix B).
    kind: "linear", "softplus" or "difference", as for ``infonce`` (the difference kind ignores ``precision``)."""
    _require_cuda(pred, targets)
    lib = _lib.load()
    if pred.dtype != torch.float32 or targets.dtype != torch.float32:
        raise _lib.CpcError("infonce_validate expects fp32 tensors")
    b, k, e = pred.shape
    if tuple(targets.shape) != (b, e, k):
        raise ValueError("targets must be (B, E, K) = %s, got %s" % ((b, e, k), tuple(targets.shape)))
    pred = pred.detach().contiguous()
    targets = targets.detach()
    p = _nce_params(pred, targets, all_steps, kind, 0.0, precision or _default_precision)
    metrics = torch.empty(2 * k + 1, dtype=torch.float32, device=pred.device)
    ws = _workspace(lib.cpc_infonce_workspace_bytes(ctypes.byref(p), 2), pred.device)
    with torch.cuda.device(pred.device):
        _call(_nce_key("cpc_infonce_validate", p), _nce_flops(p), lib.cpc_infonce_validate, _ptr(pred), _ptr(targets),
              _ptr(metrics), ctypes.byref(p), _ptr(ws), ws.numel(), _stream())
    return metrics[:k], metrics[k:2 * k], metrics[2 * k]


# --------------------------------------------------------------------------------------------------
# CQT front end (no autograd: the filterbank is frozen in training, constant_q_transform.py:145)
# --------------------------------------------------------------------------------------------------

def _cqt_params(plan, batch, n_samples, x_pitch, n_frames, mode, pool_t, eps, log_offset, norm, power):
    p = _lib.CqtParams()
    p.batch, p.n_samples, p.x_pitch = batch, n_samples, x_pitch
    p.n_bins, p.hop, p.n_frames = plan["n_bins"], plan["hop"], n_frames
    p.n_groups = len(plan["kernel_sizes"])
    for g, (ks, (lo, hi), wo) in enumerate(zip(plan["kernel_sizes"], plan["ranges"], plan["weight_offsets"])):
        p.kernel_size[g], p.bin_lo[g], p.bin_hi[g], p.weight_offset[g] = ks, lo, hi, wo
    p.mode, p.pool_t = mode, pool_t
    p.eps, p.log_offset, p.norm, p.power = eps, log_offset, norm, power
    p.flags = _lib.CQT_FLAG_NO_TENSOR if _switch("CPC_NO_TENSOR_CQT") else 0
    if _default_precision == "bf16":
        p.flags |= _lib.CQT_FLAG_HALF_OPERANDS                  # front end of the bf16 operand mode: one fp16 plane per operand
    import os
    p.flags |= (int(kernel_switches.get("CPC_CQT_ROUND", os.environ.get("CPC_CQT_ROUND", "0"))) & 0xff) << 8
    return p


def cqt_pack_filters(weights, plan):
    """The filterbank in the form the tensor-core kernel reads (scaled fp16 hi / lo planes, per-bin scales, live tap
    ranges), or None when the configuration has no tensor-core path.  Depends on the weights only: ``CQT`` caches it."""
    _require_cuda(weights)
    lib = _lib.load()
    k0 = plan["kernel_sizes"][0]
    p = _cqt_params(plan, 1, k0 + 1, k0 + 1, 1, _lib.CQT_COMPLEX, 1, 0.0, 0.0, 1.0, 1.0)
    p.flags = 0
    nbytes = lib.cpc_cqt_packed_filter_bytes(ctypes.byref(p))
    if nbytes == 0:
        return None
    packed = torch.empty(int(nbytes), dtype=torch.uint8, device=weights.device)
    with torch.cuda.device(weights.device):
        _call("cpc_cqt_pack_filters", 0.0, lib.cpc_cqt_pack_filters, _ptr(weights), _ptr(packed), ctypes.byref(p), _stream())
    return packed


def cqt_frontend(x, weights, plan, mode, phase_fixed=None, phase_scale=None, pool_t=1, eps=0.0, log_offset=0.0,
                 norm=1.0, power=1.0, packed_filters=None):
    """x (B, L) or (B,1,L) fp32 on CUDA; ``weights`` the packed filterbank; ``plan`` a dict with
    kernel_sizes / ranges / weight_offsets / hop / n_bins.  Output layout per ``mode`` (see cpc_b200.h)."""
    _require_cuda(x, weights)
    lib = _lib.load()
    if x.dim() == 3:
        if x.shape[1] != 1:
            raise ValueError("CQT expects mono input (B,1,L)")
        x = x[:, 0]
    x = x.contiguous()
    if x.dtype != torch.float32:
        raise _lib.CpcError("CQT expects fp32 audio")
    b, l = x.shape
    k0 = plan["kernel_sizes"][0]
    t = (l - 1 - k0) // plan["hop"] + 1
    if t <= 0:
        raise ValueError("input of %d samples is shorter than the CQT receptive field %d (+1)" % (l, k0))
    p = _cqt_params(plan, b, l, x.stride(0), t, mode, pool_t, eps, log_offset, norm, power)
    f = plan["n_bins"]
    if mode == _lib.CQT_COMPLEX:
        out = torch.empty((b, f, t, 2), dtype=torch.float32, device=x.device)
    elif mode == _lib.CQT_LOGPOW:
        out = torch.empty((b, 1, f, t // pool_t), dtype=torch.float32, device=x.device)
    else:
        if t < 2:
            raise ValueError("phase mode needs at least 2 CQT frames")
        out = torch.empty((b, 2, f, (t - 1) // pool_t), dtype=torch.float32, device=x.device)
    ws = _workspace(lib.cpc_cqt_workspace_bytes(ctypes.byref(p)), x.device)
    with torch.cuda.device(x.device):
        taps = sum(2 * (hi - lo) * ks for ks, (lo, hi) in zip(plan["kernel_sizes"], plan["ranges"]))
        c_out = 2 if mode == _lib.CQT_LOGPOW_PHASE else (2 if mode == _lib.CQT_COMPLEX else 1)
        _call("cpc_cqt_fwd b%d L%d T%d mode%d" % (b, l, t, mode), 2.0 * taps * b * t, lib.cpc_cqt_fwd_ex, _ptr(x),
              _ptr(weights), _ptr(packed_filters), _ptr(phase_fixed), _ptr(phase_scale), _ptr(out), ctypes.byref(p), _ptr(ws),
              ws.numel() if ws is not None else 0, _stream(), nbytes=4.0 * b * l + 4.0 * out.numel())
    return out

"""Torch-tensor wrappers over the C ABI (include/marconet_b200.h).

PyTorch is plumbing here: it owns device memory and the current CUDA stream; every
computation below is a kernel from libmarconet_b200.so.  Activations are NHWC fp32 views
``[N, H, W, C]`` with ``stride(-1) == 1`` whose pixel stride (``cs``) may exceed C (channel
slices of a concatenation buffer).
"""
import ctypes

import torch

from . import _lib
from ._lib import (ACT_GELU, ACT_LRELU02, ACT_NONE, ACT_RELU, ACT_RSQRT_EPS, ACT_SIGMOID, ACT_TANH,  # noqa: F401
                   PREC_BF16X3_TC, PREC_F16X1_TC, PREC_F16X3_TC, PREC_FP32_SIMT, ConvParams, Window)

import os as _os
import threading as _threading

_WS = {}
_WS_BYTES = 96 << 20
# per-thread launch context (graph.py captures per thread; two host threads must never see each other's scratch or error flag)
_TLS = _threading.local()
# 0 fp32 CUDA-core, 1 fp16x3 tcgen05 (default: parity-grade tensor-core path), 2 bf16x3 tcgen05, 3 fp16x1 tcgen05 (not parity grade)
_DEFAULT_PRECISION = int(_os.environ.get("MN_PRECISION", PREC_F16X3_TC))
LAUNCHES = 0   # number of C-ABI kernel-launching calls issued (bench.py reports it)


def set_default_precision(p):
    global _DEFAULT_PRECISION
    _DEFAULT_PRECISION = int(p)


def graph_key():
    """Everything process-global that a captured CUDA graph of this library bakes in."""
    return (_DEFAULT_PRECISION, PLAN_VERSION, MAX_CTAS, FUSE_GN)


def graphs_allowed():
    """Module-level graph replay is off inside another capture, inside ops.deferred_checks (GraphedLines owns the step then) and
    while a calibration records per-layer statistics."""
    return (MODULE_GRAPHS and getattr(_TLS, "deferred_flag", None) is None and getattr(_TLS, "calib", None) is None
            and not torch.cuda.is_current_stream_capturing())


MODULE_GRAPHS = _os.environ.get("MN_MODULE_GRAPHS", "1") != "0"


def set_max_ctas(n):
    """Cap the persistent conv kernels at n CTAs (0 = all SMs); returns the previous cap."""
    global MAX_CTAS
    MAX_CTAS = int(n)
    return _lib.load().mn_set_max_ctas(int(n))


def default_precision():
    return _DEFAULT_PRECISION


def _stream():
    """The current stream of the CURRENT device.  Every wrapper checks (``_require_cuda``) that its tensors live on the current
    device, and the module forwards switch to their input's device (``torch.cuda.device(x.device)``), so a model on cuda:1 driven
    from a process whose current device is cuda:0 launches on cuda:1's stream, never on cuda:0's with cuda:1 pointers."""
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def on_device(t):
    """Context manager: make ``t``'s device current (stream, SM count, dynamic-smem attributes all follow the current device)."""
    return torch.cuda.device(t.device)


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _require_cuda(t, name):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"marconet_b200: {name} must be a CUDA tensor (there is no CPU path)")
    if t.dtype != torch.float32:
        raise RuntimeError(f"marconet_b200: {name} must be float32, got {t.dtype}")
    if t.device.index != torch.cuda.current_device():
        raise RuntimeError(f"marconet_b200: {name} lives on {t.device} but the current CUDA device is cuda:{torch.cuda.current_device()}; "
                           f"call through the module API (it switches devices) or wrap the call in torch.cuda.device(...)")


def nhwc_info(t, name="tensor"):
    """(N, H, W, C, cs) of an NHWC view; verifies the stride pattern."""
    _require_cuda(t, name)
    if t.dim() != 4:
        raise RuntimeError(f"{name}: expected 4-D NHWC view, got {tuple(t.shape)}")
    n, h, w, c = t.shape
    sn, sh, sw, sc = t.stride()
    cs = sw if w > 1 else (sh if h > 1 else (sn if n > 1 else c))
    ok = (sc == 1 or c == 1) and (w == 1 or sw == cs) and (h == 1 or sh == w * cs) and (n == 1 or sn == h * w * cs)
    if not ok:
        raise RuntimeError(f"{name}: not a dense NHWC view (shape {tuple(t.shape)}, strides {t.stride()})")
    return n, h, w, c, cs


def workspace(device):
    """Split-K scratch of the conv kernels: one per device (single stream, like the reference scripts) unless a caller that runs
    convolutions on a second stream installs its own with ``use_workspace`` (per host thread)."""
    ov = getattr(_TLS, "ws_override", None)
    if ov is not None:
        return ov
    key = device.index if device.index is not None else torch.cuda.current_device()
    ws = _WS.get(key)
    if ws is None:
        ws = torch.empty(_WS_BYTES // 4, dtype=torch.float32, device=device)
        _WS[key] = ws
    return ws


class use_workspace:
    """Context manager: convolutions launched inside use ``ws`` (fp32 CUDA tensor) as their split-K scratch, so that they can run
    on another stream concurrently with convolutions that use the per-device scratch."""

    def __init__(self, ws):
        self.ws, self.prev = ws, None

    def __enter__(self):
        self.prev = getattr(_TLS, "ws_override", None)
        _TLS.ws_override = self.ws
        return self.ws

    def __exit__(self, *exc):
        _TLS.ws_override = self.prev
        return False


PLAN = {}     # layer name -> (precision or None, x_scale): the per-layer precision plan of this process (pipeline.tune_precision)
PLAN_VERSION = 0   # bumped whenever a layer's plan changes: captured CUDA graphs bake the plan in and key on it
MAX_CTAS = 0       # mirror of mn_set_max_ctas (grid sizes are baked into captured graphs)


class ConvWeight:
    """A conv/linear weight in kernel layout: fp32 K-major [KH*KW*Cin, Cout] plus (lazily) the hi/lo 16-bit
    planes [taps][Cout][Cin] the tcgen05 path consumes (mn_conv_pack_weights_tc).

    Per-layer precision plan (SURVEY 8f n4; set by pipeline.tune_precision or by the range guard):
      ``precision``  None = the process default, else one of PREC_* for this layer;
      ``x_scale``    power of two applied to the layer's INPUT inside the kernel before the fp16 hi/lo split and undone
                     exactly in the epilogue, so that |x * x_scale| stays inside fp16's range (mn_conv_params.x_scale)."""

    __slots__ = ("w", "taps", "cin", "cout", "_tc", "name", "precision", "x_scale", "tag", "__weakref__")
    _next_tag = 1
    _by_tag = {}

    def __init__(self, w, taps, name=None):
        import weakref
        self.w = w
        self.taps = taps
        self.cin = w.shape[0] // taps
        self.cout = w.shape[1]
        self._tc = {}
        self.tag = ConvWeight._next_tag
        ConvWeight._next_tag += 1
        self.name = name or f"conv#{self.tag}[{taps}x{self.cin}->{self.cout}]"
        self.precision, self.x_scale = PLAN.get(self.name, (None, 1.0))      # plans survive re-packing (keyed by layer name)
        ConvWeight._by_tag[self.tag] = weakref.ref(self)

    def set_plan(self, precision=None, x_scale=None):
        """Set this layer's precision / input scale and remember it under the layer's name (ops.PLAN)."""
        if precision is not None:
            self.precision = int(precision)
        if x_scale is not None:
            self.x_scale = float(x_scale)
        PLAN[self.name] = (self.precision, self.x_scale)
        global PLAN_VERSION
        PLAN_VERSION += 1

    @classmethod
    def from_tag(cls, tag):
        r = cls._by_tag.get(int(tag))
        return None if r is None else r()

    @property
    def shape(self):
        return self.w.shape

    def tc_capable(self):
        return self.cin % 64 == 0 and self.cout % 64 == 0

    def tc(self, precision):
        key = PREC_BF16X3_TC if precision == PREC_BF16X3_TC else PREC_F16X3_TC
        got = self._tc.get(key)
        if got is None:
            n = self.taps * self.cin * self.cout
            hi = torch.empty(n, dtype=torch.int16, device=self.w.device)
            lo = torch.empty(n, dtype=torch.int16, device=self.w.device)
            sc = torch.empty(2, dtype=torch.float32, device=self.w.device)
            with torch.cuda.device(self.w.device):
                _lib.check(_lib.load().mn_conv_pack_weights_tc(_ptr(self.w), self.taps, self.cin, self.cout, key, _ptr(hi), _ptr(lo),
                                                               _ptr(sc), _stream()), "mn_conv_pack_weights_tc")
            got = (hi, lo, sc)
            self._tc[key] = got
        return got


# ---- fp16-range guard (ADVICE r1 / VERDICT r1 2.iii) ------------------------------------------------------------------
# The default tensor-core precision splits fp32 operands into fp16 hi/lo pairs: an activation with |x * x_scale| >= 65504 would
# become Inf.  Every tensor-core conv is launched with a pointer to a per-device flag in PINNED HOST memory; the operand-split
# stage stores the layer's tag into it when an element leaves the range (or is Inf/NaN).  The host reads the flag without any
# CUDA call: at the start of every module forward (``poll_range``: the offending layer is re-routed to the bf16 split, which has
# fp32's exponent range, and a warning names it -- the overflowed call's own output contains Inf/NaN, never a silently wrong
# number) and in ``check_range`` (raises FloatingPointError; GraphedLines.check and pipeline.restore_lines call it after their
# synchronisation, the latter re-runs the step once with the new plan).
_RANGE_FLAGS = {}
_RANGE_SLOTS = 2048
RANGE_EVENTS = []        # (layer name, action) log of re-routes, newest last


def range_flags(device):
    """Per-device int32[_RANGE_SLOTS] in pinned host memory; slot tag % _RANGE_SLOTS belongs to the layer with that tag."""
    key = device.index if device.index is not None else torch.cuda.current_device()
    f = _RANGE_FLAGS.get(key)
    if f is None:
        f = torch.zeros(_RANGE_SLOTS, dtype=torch.int32).pin_memory()
        _RANGE_FLAGS[key] = f
    return f


def poll_range(device, reroute=True):
    """Non-synchronising look at the device's range flags.  Returns the offending ConvWeights (empty list: none) and clears the
    flags; with ``reroute`` every such layer is switched to the bf16 hi/lo split for all later calls."""
    f = _RANGE_FLAGS.get(device.index if device.index is not None else torch.cuda.current_device())
    if f is None:
        return []
    arr = f.numpy()
    if not arr.any():
        return []
    tags = [int(t) for t in arr[arr != 0]]
    arr[:] = 0
    hits = []
    import warnings
    for tag in tags:
        cw = ConvWeight.from_tag(tag)
        if cw is None:
            continue
        hits.append(cw)
        if not reroute:
            continue
        if cw.precision == PREC_BF16X3_TC:      # already on the wide-range split: the input itself held Inf / NaN
            RANGE_EVENTS.append((cw.name, "non-finite input"))
            warnings.warn(f"marconet_b200: non-finite values reached conv layer {cw.name}")
        else:
            cw.set_plan(precision=PREC_BF16X3_TC)
            RANGE_EVENTS.append((cw.name, "rerouted to bf16x3"))
            warnings.warn(f"marconet_b200: |activation * {cw.x_scale:g}| >= 65504 at conv layer {cw.name}: the fp16 hi/lo split "
                          f"overflowed (that call's output holds Inf/NaN); the layer now uses the bf16 split (MN_PREC_BF16X3_TC). "
                          f"Run pipeline.tune_precision() for a calibrated per-layer plan.")
    return hits


def check_range(device):
    """Raise FloatingPointError when a tensor-core conv saw an operand outside its representable range since the last
    poll.  The caller must have synchronised with the work it asks about."""
    hits = poll_range(device)
    if hits:
        names = ", ".join(cw.name for cw in hits[:6]) + (" ..." if len(hits) > 6 else "")
        raise FloatingPointError(f"marconet_b200: fp16 operand range exceeded (or non-finite input) at conv layer(s) {names}; they "
                                 f"have been re-routed to the bf16 split -- re-run the step")


class calibration:
    """Context manager: every tensor-core conv launched inside records max |x * x_scale| of its input (mn_conv_params.x_absmax)
    and, with ``compare=True``, its relative max-abs error against the exact fp32 kernel for both split formats.
    ``results()`` (synchronises) -> {ConvWeight: dict(absmax=..., err_f16x3=..., err_bf16x3=..., out_absmax=...)}."""

    SLOTS = 4096

    def __init__(self, device, compare=False):
        self.device, self.compare = torch.device(device), compare
        self.buf = torch.zeros(self.SLOTS, dtype=torch.float32, device=self.device)
        self.slots, self.errs, self.prev = {}, {}, None

    def __enter__(self):
        self.prev = getattr(_TLS, "calib", None)
        _TLS.calib = self
        return self

    def __exit__(self, *exc):
        _TLS.calib = self.prev
        return False

    def slot(self, cw):
        i = self.slots.get(cw)
        if i is None:
            i = len(self.slots)
            if i >= self.SLOTS:
                raise RuntimeError("calibration: too many layers")
            self.slots[cw] = i
        return self.buf[i:i + 1]

    def results(self):
        torch.cuda.synchronize(self.device)
        host = self.buf.cpu()
        out = {}
        for cw, i in self.slots.items():
            rec = dict(absmax=float(host[i]) / cw.x_scale)
            for k, v in self.errs.get(cw, {}).items():
                rec[k] = max(float(t) for t in v)
            out[cw] = rec
        return out


TC_FALLBACKS = {}      # shape key -> (layer name, GFLOP, reason): convs that a tensor-core default ran on the fp32 CUDA-core kernel


def _note_fallback(cw, key, flop, reason):
    """A tensor-core precision was the default but this conv runs on the exact fp32 kernel (unsupported geometry: Cin/Cout not
    multiples of 64, stride != 1, tiny launch ...).  Logged ONCE per shape so that a checkpoint with different channel counts does
    not quietly run 6x slower (VERDICT r1); ``ops.TC_FALLBACKS`` keeps the list, bench.py reports it."""
    if key in TC_FALLBACKS:
        return
    name = cw.name if cw is not None else "unnamed"
    TC_FALLBACKS[key] = (name, flop / 1e9, reason)
    import logging
    logging.getLogger("marconet_b200").info("conv %s %s runs on the fp32 CUDA-core kernel: %s", name, key, reason)


# fused GroupNorm(+swish) input transform of the tcgen05 conv (MN_FUSE_GN): "1" (default) every layer that kernel runs, "0" never
# (mn_groupnorm_apply writes a normalised copy first), "auto" only the layers with 128-wide tiles (Cout % 128 == 0)
FUSE_GN = {"0": 0, "1": 1, "auto": 2, "2": 2}.get(_os.environ.get("MN_FUSE_GN", "1"), 1)


def _fuse_gn(cout):
    return FUSE_GN == 1 or (FUSE_GN == 2 and cout % 128 == 0)
TC_MIN_FLOP = 3.0e7    # tiny launches are latency-bound either way and stay on the exact fp32 path


def conv2d(x, w, kh, kw, stride=(1, 1), pad=(0, 0), bias=None, out_scale=None, residual=None,
           res_broadcast=False, act=ACT_NONE, gain=1.0, out=None, out2=None, y2_scale=None,
           valid_w=None, precision=None, want_y=True, split_k=0, gn=None, gn_fuse=None, out2_ptrs=None, gn_stats=False):
    """mn_conv2d_nhwc.  ``w`` is the packed [KH*KW*Cin, Cout] matrix.  Returns y (or (y, y2)).
    ``gn=(mean_rstd, gamma, beta)``: the conv input is swish(GroupNorm(x)); fused into the tcgen05 kernel's operand-split
    stage when ``gn_fuse`` is true and that kernel runs the layer, otherwise applied by mn_groupnorm_apply first.
    (Default on since the fused instantiation runs four lanes per halo row with the GroupNorm constants in registers: all eight
    normalise passes gone, 1.3 % per line on the same box, profiles/r2_split_gn_ab.txt; its first form -- one lane per row, per-row
    global loads of mean / rstd -- measured 8.7 vs 7.1 ms.)
    ``gn_stats=True``: also return the GroupNorm statistics (mean / rstd [N, Cout/32, 2]) of the OUTPUT, for the GroupNorm that
    follows this conv (networks.py:508-512): accumulated by the tcgen05 kernel's epilogue (mn_conv_params.gn_stats_out, no read
    pass over y) when that kernel runs the layer, by mn_groupnorm_stats otherwise.  Returns (y, mean_rstd)."""
    global LAUNCHES
    lib = _lib.load()
    n, h, wd, cin, x_cs = nhwc_info(x, "x")
    cw = w if isinstance(w, ConvWeight) else None
    if cw is not None:
        w = cw.w
    cout = w.shape[1]
    if w.shape[0] != kh * kw * cin:
        raise RuntimeError(f"conv2d: packed weight has {w.shape[0]} rows, expected {kh * kw * cin}")
    oh = (h + 2 * pad[0] - kh) // stride[0] + 1
    ow = (wd + 2 * pad[1] - kw) // stride[1] + 1
    p = ConvParams()
    p.x = x.data_ptr(); p.N = n; p.H = h; p.W = wd; p.Cin = cin; p.x_cs = x_cs
    p.w = w.data_ptr(); p.KH = kh; p.KW = kw; p.stride_h, p.stride_w = stride; p.pad_h, p.pad_w = pad; p.Cout = cout
    y = None
    if want_y:
        y = out if out is not None else torch.empty((n, oh, ow, cout), dtype=torch.float32, device=x.device)
        yn, yh, yw, yc, y_cs = nhwc_info(y, "out")
        if (yn, yh, yw, yc) != (n, oh, ow, cout):
            raise RuntimeError(f"conv2d: out has shape {tuple(y.shape)}, expected {(n, oh, ow, cout)}")
        p.y = y.data_ptr(); p.y_cs = y_cs
    y2 = None
    if out2_ptrs is not None:
        # second output scattered through per-sample base pointers (int64 device tensor [N], possibly PEER-GPU addresses):
        # mn_conv_params.y2_ptrs; dense [OH, OW, Cout] blocks.  Nothing local is allocated for it.
        if out2 is not None or out2_ptrs.dtype != torch.int64 or not out2_ptrs.is_cuda or out2_ptrs.numel() != n or not out2_ptrs.is_contiguous():
            raise RuntimeError("conv2d: out2_ptrs must be a contiguous int64 CUDA tensor with one pointer per sample (and out2 unset)")
        p.y2 = out2_ptrs.data_ptr(); p.y2_cs = cout; p.y2_ptrs = out2_ptrs.data_ptr()
        if y2_scale is not None:
            p.y2_scale = y2_scale.data_ptr(); p.y2_scale_stride = y2_scale.stride(0)
    if out2 is not None:
        y2 = out2 if isinstance(out2, torch.Tensor) else torch.empty((n, oh, ow, cout), dtype=torch.float32, device=x.device)
        _, _, _, _, y2_cs = nhwc_info(y2, "out2")
        p.y2 = y2.data_ptr(); p.y2_cs = y2_cs
        if y2_scale is not None:
            p.y2_scale = y2_scale.data_ptr(); p.y2_scale_stride = y2_scale.stride(0)
    if bias is not None:
        p.bias = bias.data_ptr()
    if out_scale is not None:
        p.out_scale = out_scale.data_ptr(); p.out_scale_stride = out_scale.stride(0)
    if residual is not None:
        rinfo = nhwc_info(residual, "residual")
        p.residual = residual.data_ptr(); p.res_cs = rinfo[4]; p.res_broadcast_n = 1 if res_broadcast else 0
    p.act = act; p.act_gain = gain
    if valid_w is not None:
        p.valid_w = valid_w.data_ptr()
    ws = workspace(x.device)
    p.workspace = ws.data_ptr(); p.workspace_bytes = ws.numel() * 4
    p.split_k = split_k
    prec = precision if precision is not None else (cw.precision if (cw is not None and cw.precision is not None) else _DEFAULT_PRECISION)
    gn_fused = False
    if prec != PREC_FP32_SIMT:
        flop = 2.0 * n * oh * ow * cout * kh * kw * cin
        why = None                            # why the tensor-core kernel does not run this conv
        if precision is None and flop < TC_MIN_FLOP:
            why = f"below TC_MIN_FLOP ({flop / 1e6:.1f} MFLOP)"
        elif cw is None or not cw.tc_capable():
            why = "Cin or Cout is not a multiple of 64"
        elif stride != (1, 1):
            why = "stride != 1"
        elif not lib.mn_conv2d_tc_supported(ctypes.byref(p)):
            why = lib.mn_last_error().decode(errors="replace") or "unsupported geometry"     # the kernel's planner says why
        if why is None:
            hi, lo, sc = cw.tc(prec)
            p.w_tc_hi = hi.data_ptr(); p.w_tc_lo = lo.data_ptr(); p.w_tc_scale = sc.data_ptr()
            p.x_scale = cw.x_scale
            p.range_flag = range_flags(x.device).data_ptr() + 4 * (cw.tag % _RANGE_SLOTS); p.range_tag = cw.tag
            calib = getattr(_TLS, "calib", None)
            if calib is not None:
                p.x_absmax = calib.slot(cw).data_ptr()
            if gn is not None and h * wd >= 128 and (_fuse_gn(cout) if gn_fuse is None else gn_fuse):   # one sample per 128-pixel tile
                p.gn_mean_rstd = gn[0].data_ptr(); p.gn_gamma = gn[1].data_ptr(); p.gn_beta = gn[2].data_ptr(); p.gn_swish = 1
                gn_fused = True
        elif precision is not None:
            raise RuntimeError("conv2d: tensor-core precision requested explicitly but this layer/shape is not supported: " + why)
        else:
            prec = PREC_FP32_SIMT
            _note_fallback(cw, (n, h, wd, cin, cout, kh, kw, stride), flop, why)
    p.precision = prec
    stats_ws = None
    if gn_stats and prec != PREC_FP32_SIMT and oh * ow >= 128 and cout % 32 == 0 and y is not None and out2_ptrs is None:
        stats_ws = torch.zeros((n * (cout // 32) * 2,), dtype=torch.float64, device=x.device)
        p.gn_stats_out = stats_ws.data_ptr()
    if gn is not None and not gn_fused:      # no fused kernel for this layer: normalise into a temporary first
        xg = groupnorm_apply(x, gn[0], gn[1], gn[2], valid_w=valid_w)
        p.x = xg.data_ptr(); p.x_cs = xg.shape[3]
    _lib.check(lib.mn_conv2d_nhwc(ctypes.byref(p), _stream()), "mn_conv2d_nhwc")
    LAUNCHES += 1
    calib = getattr(_TLS, "calib", None)
    if calib is not None and calib.compare and cw is not None and prec != PREC_FP32_SIMT and precision is None:
        # tuning tool only (pipeline.tune_precision): the same layer through the exact fp32 kernel and both split formats
        _TLS.calib = None
        try:
            opts = dict(stride=stride, pad=pad, bias=bias, out_scale=out_scale, residual=residual, res_broadcast=res_broadcast, act=act,
                        gain=gain, valid_w=valid_w, split_k=split_k, gn=gn)
            ref = conv2d(x, cw, kh, kw, precision=PREC_FP32_SIMT, **opts)
            scale = ref.abs().max().clamp_min(1e-30)
            rec = calib.errs.setdefault(cw, {})
            rec.setdefault("out_absmax", []).append(scale)
            for name, cand in (("err_f16x3", PREC_F16X3_TC), ("err_bf16x3", PREC_BF16X3_TC)):
                got = conv2d(x, cw, kh, kw, precision=cand, **opts)
                rec.setdefault(name, []).append(torch.nan_to_num((got - ref).abs().max() / scale, nan=float("inf")))
        finally:
            _TLS.calib = calib
    if gn_stats:
        if stats_ws is not None:
            mr = torch.empty((n, cout // 32, 2), dtype=torch.float32, device=x.device)
            _lib.check(lib.mn_groupnorm_finalize(_ptr(stats_ws), n, oh, ow, cout, 32, 1e-6, _ptr(valid_w), _ptr(mr), _stream()), "mn_groupnorm_finalize")
            LAUNCHES += 2
        else:
            mr = groupnorm_stats(y, valid_w=valid_w)
        return y, mr
    if y2 is not None:
        return (y, y2) if want_y else y2
    return y


def linear(x2d, w, bias=None, act=ACT_NONE, gain=1.0, residual=None, out=None, precision=None):
    """nn.Linear as a 1x1 conv on [M,1,1,K]; ``w`` packed [K, Cout]; x2d: [M, K] contiguous."""
    global LAUNCHES
    m, k = x2d.shape
    wt = w.w if isinstance(w, ConvWeight) else w
    nout = wt.shape[1]
    if m <= 64 and k % 32 == 0 and nout % 16 == 0 and precision is None and x2d.is_contiguous() and \
            (residual is None or residual.is_contiguous()):
        y = out if out is not None else torch.empty((m, nout), dtype=torch.float32, device=x2d.device)
        _lib.check(_lib.load().mn_linear_small_m(_ptr(x2d), _ptr(wt), _ptr(bias), _ptr(residual), _ptr(y), m, k, nout, act, gain,
                                                 _stream()), "mn_linear_small_m")
        LAUNCHES += 1
        return y
    res = None if residual is None else residual.reshape(m, 1, 1, -1)
    o = None if out is None else out.reshape(m, 1, 1, -1)
    y = conv2d(x2d.reshape(m, 1, 1, k), w, 1, 1, bias=bias, act=act, gain=gain, residual=res, out=o, precision=precision)
    return y.reshape(m, -1)


def patch_embed(feat, w, bias, pe):
    """TextViT patch embedding on the NHWC feature map in place (textvit_arch.py:33-36,68-69):
    feat [B, 8, 8*T, C] -> tokens [B*T, D] = Linear(rearrange(feat, 'b (p1) (t p2) c -> b t (p1 p2 c)')) + pe[T, D].
    ``w`` is the packed [8*8*C, D] weight (K order p1, p2, c)."""
    global LAUNCHES
    b, fh, fw, c, cs = nhwc_info(feat, "feat")
    if fh != 8 or fw % 8 != 0 or cs != c:
        raise RuntimeError("patch_embed: expects a dense [B, 8, 8*T, C] feature map")
    t = fw // 8
    k, d = w.shape
    if k != 64 * c or t > 64 or tuple(pe.shape) != (t, d):
        raise RuntimeError("patch_embed: weight / positional embedding do not match the feature map")
    y = torch.empty((b * t, d), dtype=torch.float32, device=feat.device)
    ws = workspace(feat.device)         # outer K slices (deep K, few column tiles): partial tiles + a deterministic reduce kernel
    _lib.check(_lib.load().mn_linear_small_m_ws(_ptr(feat), 8 * c, 8 * fw * c, 8 * c, fw * c, _ptr(w), _ptr(bias), _ptr(pe), 0, _ptr(y),
                                                b, t, k, d, ACT_NONE, 1.0, _ptr(ws), ws.numel() * 4, _stream()), "mn_linear_small_m_ws")
    LAUNCHES += 2
    return y


def pixelnorm(x):
    global LAUNCHES
    _require_cuda(x, "x")
    y = torch.empty_like(x)
    _lib.check(_lib.load().mn_pixelnorm(_ptr(x), _ptr(y), x.shape[0], x.shape[1], _stream()), "mn_pixelnorm")
    LAUNCHES += 1
    return y


# ---- deferred error checks (CUDA-graph capture / pipelined callers, SURVEY 8f n1) -----------------------------------
# The module API raises on a bad label or an empty character window BEFORE launching, which costs a device->host round
# trip per call.  Inside ``deferred_checks(flag)`` the same conditions are evaluated by device kernels that OR a bit into
# ``flag`` (int32[1] on the device: bit 0 = label out of range, bit 1 = empty window); the caller reads it with the results.
ERR_LABEL, ERR_WINDOW = 1, 2


class deferred_checks:
    def __init__(self, flag):
        if flag is not None and (flag.dtype != torch.int32 or not flag.is_cuda or flag.numel() != 1):
            raise RuntimeError("deferred_checks: flag must be an int32[1] CUDA tensor")
        self.flag, self.prev = flag, None

    def __enter__(self):
        self.prev = getattr(_TLS, "deferred_flag", None)
        _TLS.deferred_flag = self.flag
        return self.flag

    def __exit__(self, *exc):
        _TLS.deferred_flag = self.prev
        return False


def deferred_flag():
    return getattr(_TLS, "deferred_flag", None)


def raise_deferred(flag_value):
    """Turn a flag value read back from the device into the exception the eager path raises."""
    if flag_value & ERR_LABEL:
        raise IndexError("character label out of range (reference: empty embedding slice, networks.py:211)")
    if flag_value & ERR_WINDOW:
        raise RuntimeError("empty character window (the reference fails on the empty slice at networks.py:443)")


def check_labels(labels_dev, classes, flag):
    """labels_dev: int64 [n] on the device -> clamped copy; raises bit 0 of ``flag`` on the device when out of range."""
    global LAUNCHES
    n = labels_dev.numel()
    out = torch.empty_like(labels_dev)
    _lib.check(_lib.load().mn_check_labels(_ptr(labels_dev), _ptr(out), n, classes, _ptr(flag), _stream()), "mn_check_labels")
    LAUNCHES += 1
    return out


def char_windows(locs_dev, line_first_dev, counts, width, half, flag):
    """Device restatement of models.networks.char_windows: returns (win int32[Nc,4], valid int32[Nc], owner int32[B,W])."""
    global LAUNCHES
    _require_cuda(locs_dev, "locs")
    if locs_dev.dtype != torch.float32 or locs_dev.dim() != 2 or locs_dev.stride(1) != 1:
        raise RuntimeError("char_windows: locs must be fp32 [B, 2n] with unit inner stride")
    b, nc = len(counts), sum(counts)
    if locs_dev.shape[0] < b or (counts and locs_dev.shape[1] < 2 * max(counts)):
        raise RuntimeError("char_windows: locs has fewer entries than characters")
    dev = locs_dev.device
    win = torch.empty((nc, 4), dtype=torch.int32, device=dev)
    valid = torch.empty((nc,), dtype=torch.int32, device=dev)
    owner = torch.empty((b, width), dtype=torch.int32, device=dev)
    _lib.check(_lib.load().mn_char_windows(_ptr(locs_dev), locs_dev.stride(0), _ptr(line_first_dev), b, max(counts), width, half,
                                           _ptr(win), _ptr(valid), _ptr(owner), _ptr(flag), _stream()), "mn_char_windows")
    LAUNCHES += 1
    return win, valid, owner


def char_segment_styles(w, locs_dev, line_first_dev, counts, width, segs, seg_w=512):
    """mn_char_segment_styles: style row of every character of B wide lines, taken from the encoder segment that holds the
    character's 32-level window centre.  ``w``: [B*segs, D] (row b*segs + s = segment s of line b); ``locs_dev``: fp32 [B, >= 2n]
    on the device; ``line_first_dev``: device int32[B+1] prefix sums of ``counts``.  Returns (styles [Nc, D], seg int32 [Nc])."""
    global LAUNCHES
    _require_cuda(w, "w")
    _require_cuda(locs_dev, "locs")
    b, nc = len(counts), sum(counts)
    if w.dim() != 2 or w.stride(1) != 1 or w.shape[0] != b * segs:
        raise RuntimeError(f"char_segment_styles: w must be [{b * segs}, D] with unit inner stride, got {tuple(w.shape)}")
    if locs_dev.dim() != 2 or locs_dev.stride(1) != 1 or locs_dev.shape[0] < b or (counts and locs_dev.shape[1] < 2 * max(counts)):
        raise RuntimeError("char_segment_styles: locs must be fp32 [B, >= 2n] with unit inner stride")
    if line_first_dev.dtype != torch.int32 or not line_first_dev.is_cuda or line_first_dev.numel() != b + 1:
        raise RuntimeError("char_segment_styles: line_first must be a device int32[B+1] tensor")
    styles = torch.empty((nc, w.shape[1]), dtype=torch.float32, device=w.device)
    seg = torch.empty((nc,), dtype=torch.int32, device=w.device)
    if nc == 0:
        return styles, seg
    _lib.check(_lib.load().mn_char_segment_styles(_ptr(w), w.stride(0), _ptr(locs_dev), locs_dev.stride(0), _ptr(line_first_dev), b,
                                                  max(counts), width, seg_w, segs, w.shape[1], _ptr(styles), styles.stride(0), _ptr(seg),
                                                  _stream()), "mn_char_segment_styles")
    LAUNCHES += 1
    return styles, seg


def select_text(emb, labels_dev, s, n, l):
    """emb: [classes, C]; labels_dev: int64 [n*l] on device; s: [n, C] view (row stride s.stride(0)) or None."""
    global LAUNCHES
    c = emb.shape[1]
    out = torch.empty((n, 4, 4 * l, c), dtype=torch.float32, device=emb.device)
    _lib.check(_lib.load().mn_select_text(_ptr(emb), _ptr(labels_dev), _ptr(s), 0 if s is None else s.stride(0),
                                          _ptr(out), n, l, c, _stream()), "mn_select_text")
    LAUNCHES += 1
    return out


def demod(s, wsq):
    """s: [N, Cin] view; wsq: [Cin, Cout] -> [N, Cout]."""
    global LAUNCHES
    n, cin = s.shape
    cout = wsq.shape[1]
    out = torch.empty((n, cout), dtype=torch.float32, device=s.device)
    _lib.check(_lib.load().mn_demod(_ptr(s), s.stride(0), _ptr(wsq), _ptr(out), n, cin, cout, _stream()), "mn_demod")
    LAUNCHES += 1
    return out


def make_demod_table(entries, device):
    """entries: [(wsq tensor [cin,cout], s_off, out_off)] -> (device byte tensor holding mn_demod_desc[], n, max_cout, total_out)."""
    import numpy as np
    arr = (_lib.DemodDesc * len(entries))()
    mx = 0
    for i, (wsq, s_off, out_off) in enumerate(entries):
        arr[i].wsq = wsq.data_ptr(); arr[i].s_off = s_off; arr[i].cin = wsq.shape[0]; arr[i].cout = wsq.shape[1]; arr[i].out_off = out_off
        mx = max(mx, wsq.shape[1])
    raw = torch.from_numpy(np.frombuffer(bytes(arr), dtype=np.uint8).copy()).to(device)
    return raw, len(entries), mx


def demod_batched(s_all, table, out_total):
    """One launch for every styled conv's demodulation vector; returns [N, out_total]."""
    global LAUNCHES
    raw, n_layers, mx = table
    n = s_all.shape[0]
    out = torch.empty((n, out_total), dtype=torch.float32, device=s_all.device)
    _lib.check(_lib.load().mn_demod_batched(_ptr(s_all), s_all.stride(0), _ptr(raw), n_layers, mx, _ptr(out), out_total, n, _stream()),
               "mn_demod_batched")
    LAUNCHES += 1
    return out


def resample_modulate(x, s=None, up=False, out=None):
    global LAUNCHES
    n, h, w, c, x_cs = nhwc_info(x, "x")
    oh, ow = (2 * h, 2 * w) if up else (h, w)
    y = out if out is not None else torch.empty((n, oh, ow, c), dtype=torch.float32, device=x.device)
    yn, yh, yw, yc, y_cs = nhwc_info(y, "out")
    if (yn, yh, yw, yc) != (n, oh, ow, c):
        raise RuntimeError(f"resample_modulate: out has shape {tuple(y.shape)}, expected {(n, oh, ow, c)}")
    _lib.check(_lib.load().mn_resample_modulate(_ptr(x), x_cs, _ptr(y), y_cs, _ptr(s), 0 if s is None else s.stride(0),
                                                n, h, w, c, 1 if up else 0, _stream()), "mn_resample_modulate")
    LAUNCHES += 1
    return y


def torgb(x, s, w, bias, skip=None):
    global LAUNCHES
    n, h, wd, c, x_cs = nhwc_info(x, "x")
    out = torch.empty((n, h, wd, 3), dtype=torch.float32, device=x.device)
    _lib.check(_lib.load().mn_torgb(_ptr(x), x_cs, _ptr(s), s.stride(0), _ptr(w), _ptr(bias), _ptr(skip), _ptr(out),
                                    n, h, wd, c, _stream()), "mn_torgb")
    LAUNCHES += 1
    return out


def groupnorm_swish(x, gamma, beta, cpg=32, eps=1e-6, swish=True, valid_w=None, out=None):
    global LAUNCHES
    n, h, w, c, x_cs = nhwc_info(x, "x")
    y = out if out is not None else torch.empty((n, h, w, c), dtype=torch.float32, device=x.device)
    _, _, _, _, y_cs = nhwc_info(y, "out")
    stats = torch.empty((n * (c // cpg) * 3,), dtype=torch.float64, device=x.device)
    _lib.check(_lib.load().mn_groupnorm_swish(_ptr(x), x_cs, _ptr(y), y_cs, _ptr(gamma), _ptr(beta), n, h, w, c, cpg,
                                              eps, 1 if swish else 0, _ptr(valid_w), _ptr(stats), _stream()),
               "mn_groupnorm_swish")
    LAUNCHES += 3
    return y


def groupnorm_stats(x, cpg=32, eps=1e-6, valid_w=None):
    """Per (sample, group) mean / rstd [N, C/cpg, 2] of an NHWC view (mn_groupnorm_stats)."""
    global LAUNCHES
    n, h, w, c, x_cs = nhwc_info(x, "x")
    g = c // cpg
    ws = torch.empty((n * g * 2,), dtype=torch.float64, device=x.device)
    mr = torch.empty((n, g, 2), dtype=torch.float32, device=x.device)
    _lib.check(_lib.load().mn_groupnorm_stats(_ptr(x), x_cs, n, h, w, c, cpg, eps, _ptr(valid_w), _ptr(ws), _ptr(mr), _stream()),
               "mn_groupnorm_stats")
    LAUNCHES += 3
    return mr


def groupnorm_apply(x, mr, gamma, beta, cpg=32, swish=True, valid_w=None, out=None):
    global LAUNCHES
    n, h, w, c, x_cs = nhwc_info(x, "x")
    y = out if out is not None else torch.empty((n, h, w, c), dtype=torch.float32, device=x.device)
    _, _, _, _, y_cs = nhwc_info(y, "out")
    _lib.check(_lib.load().mn_groupnorm_apply(_ptr(x), x_cs, _ptr(y), y_cs, _ptr(gamma), _ptr(beta), _ptr(mr), n, h, w, c, cpg,
                                              1 if swish else 0, _ptr(valid_w), _stream()), "mn_groupnorm_apply")
    LAUNCHES += 1
    return y


def adain_concat(prior, feat, win_dev, nc, wp):
    global LAUNCHES
    pn, h, pw, c, p_cs = nhwc_info(prior, "prior")
    b, fh, w, fc, f_cs = nhwc_info(feat, "feat")
    if pn != nc or pw != wp or fh != h or fc != c:
        raise RuntimeError("adain_concat: shape mismatch")
    out = torch.empty((nc, h, wp, 2 * c), dtype=torch.float32, device=feat.device)
    stats = torch.empty((nc * c * 6,), dtype=torch.float64, device=feat.device)
    _lib.check(_lib.load().mn_adain_concat(_ptr(prior), p_cs, _ptr(feat), f_cs, _ptr(win_dev), _ptr(out), nc, h, wp, w, c,
                                           _ptr(stats), _stream()), "mn_adain_concat")
    LAUNCHES += 3
    return out


def window_scatter(feat, scale, shift, owner_dev, win_dev, wp, out=None):
    global LAUNCHES
    b, h, w, c, f_cs = nhwc_info(feat, "feat")
    y = out if out is not None else torch.empty((b, h, w, c), dtype=torch.float32, device=feat.device)
    _, _, _, _, y_cs = nhwc_info(y, "out")
    _lib.check(_lib.load().mn_window_scatter(_ptr(feat), f_cs, _ptr(scale), _ptr(shift), _ptr(owner_dev), _ptr(win_dev),
                                             _ptr(y), y_cs, b, h, w, wp, c, _stream()), "mn_window_scatter")
    LAUNCHES += 1
    return y


def swish(x):
    """x * sigmoid(x) on a CUDA tensor of any shape (reference networks.py:492-493)."""
    global LAUNCHES
    _require_cuda(x, "x")
    x = x.contiguous()
    y = torch.empty_like(x)
    _lib.check(_lib.load().mn_swish(_ptr(x), _ptr(y), x.numel(), _stream()), "mn_swish")
    LAUNCHES += 1
    return y


def calc_mean_std_4d(feat, eps=1e-5):
    """reference networks.py:518-525 on an NCHW CUDA tensor -> (mean [B,C,1,1], std [B,C,1,1]) (unbiased variance + eps)."""
    global LAUNCHES
    _require_cuda(feat, "feat")
    if feat.dim() != 4:
        raise AssertionError("The input feature should be 4D tensor.")
    b, c, h, w = feat.shape
    x = feat.contiguous()
    mean = torch.empty((b, c, 1, 1), dtype=torch.float32, device=feat.device)
    std = torch.empty((b, c, 1, 1), dtype=torch.float32, device=feat.device)
    _lib.check(_lib.load().mn_row_mean_std(_ptr(x), _ptr(mean), _ptr(std), b * c, h * w, eps, _stream()), "mn_row_mean_std")
    LAUNCHES += 1
    return mean, std


def adaptive_instance_normalization(prior_feat, lq_feat):
    """reference networks.py:528-533 on NCHW CUDA tensors with equal [B, C]."""
    global LAUNCHES
    lm, ls = calc_mean_std_4d(lq_feat)
    pm, ps = calc_mean_std_4d(prior_feat)
    if lm.shape != pm.shape:
        raise RuntimeError("adaptive_instance_normalization: prior and lq features disagree on [B, C]")
    b, c, h, w = prior_feat.shape
    x = prior_feat.contiguous()
    out = torch.empty_like(x)
    _lib.check(_lib.load().mn_adain_rows(_ptr(x), _ptr(pm), _ptr(ps), _ptr(lm), _ptr(ls), _ptr(out), b * c, h * w, _stream()), "mn_adain_rows")
    LAUNCHES += 1
    return out


def layernorm(x2d, gamma, beta, eps=1e-5):
    global LAUNCHES
    _require_cuda(x2d, "x")
    rows, dim = x2d.shape
    y = torch.empty_like(x2d)
    _lib.check(_lib.load().mn_layernorm(_ptr(x2d), _ptr(y), _ptr(gamma), _ptr(beta), rows, dim, eps, _stream()), "mn_layernorm")
    LAUNCHES += 1
    return y


def token_mix(x, gamma, beta, w, bias, eps=1e-5):
    """x: [B,T,D] contiguous -> [B,To,D]."""
    global LAUNCHES
    b, t, d = x.shape
    to = w.shape[0]
    out = torch.empty((b, to, d), dtype=torch.float32, device=x.device)
    _lib.check(_lib.load().mn_token_mix(_ptr(x), _ptr(gamma), _ptr(beta), _ptr(w), _ptr(bias), _ptr(out), b, t, to, d, eps,
                                        _stream()), "mn_token_mix")
    LAUNCHES += 1
    return out


def attention(qkv, heads=8, dh=64):
    """qkv: [B,S,3*heads*dh] contiguous -> [B,S,heads*dh]."""
    global LAUNCHES
    b, s, _ = qkv.shape
    out = torch.empty((b, s, heads * dh), dtype=torch.float32, device=qkv.device)
    _lib.check(_lib.load().mn_attention(_ptr(qkv), _ptr(out), b, s, heads, dh, dh ** -0.5, _stream()), "mn_attention")
    LAUNCHES += 1
    return out


def nchw_to_nhwc(x, out=None):
    global LAUNCHES
    _require_cuda(x, "x")
    n, c, h, w = x.shape
    x = x.contiguous()
    y = out if out is not None else torch.empty((n, h, w, c), dtype=torch.float32, device=x.device)
    _, _, _, _, y_cs = nhwc_info(y, "out")
    _lib.check(_lib.load().mn_nchw_to_nhwc(_ptr(x), _ptr(y), n, c, h, w, y_cs, _stream()), "mn_nchw_to_nhwc")
    LAUNCHES += 1
    return y


def nhwc_to_nchw(x):
    global LAUNCHES
    n, h, w, c, x_cs = nhwc_info(x, "x")
    y = torch.empty((n, c, h, w), dtype=torch.float32, device=x.device)
    _lib.check(_lib.load().mn_nhwc_to_nchw(_ptr(x), x_cs, _ptr(y), n, c, h, w, _stream()), "mn_nhwc_to_nchw")
    LAUNCHES += 1
    return y


def as_nhwc(x_nchw):
    """NCHW-shaped tensor -> NHWC view, zero-copy when the input is channels_last."""
    n, c, h, w = x_nchw.shape
    v = x_nchw.permute(0, 2, 3, 1)
    if v.is_contiguous():
        return v
    return nchw_to_nhwc(x_nchw)


def as_nchw_view(x_nhwc):
    """NHWC tensor -> NCHW-shaped view (channels_last strides); what the modules return."""
    return x_nhwc.permute(0, 3, 1, 2)


# ---- script pre/post-processing on the device (SURVEY 8f n2) ---------------------------------------------------------
def round_half_even(v):
    """cv::saturate_cast<int>(double) = cvRound: round half to even (how cv::resize derives dsize from fx, fy)."""
    return int(round(v))          # Python's round() is round-half-even on floats


def preprocess_lq(img_u8, out_h=32, out_w=512, return_resized=False):
    """test_sr.py:98-111 on the device.  img_u8: uint8 [h, w, 3] CUDA tensor (the BGR image the script reads) ->
    (lq fp32 [1, 3, out_h, out_w], resized width).  Bit-identical to OpenCV's own INTER_CUBIC + ToTensor + Normalize."""
    global LAUNCHES
    if not isinstance(img_u8, torch.Tensor) or not img_u8.is_cuda:
        raise RuntimeError("marconet_b200: img must be a CUDA tensor (there is no CPU path)")
    if img_u8.dtype != torch.uint8 or img_u8.dim() != 3 or not img_u8.is_contiguous():
        raise RuntimeError("preprocess_lq: expects a contiguous uint8 [h, w, c] image")
    h, w, cn = img_u8.shape
    fx = fy = out_h / h                                   # Python float division, like the script's fx=32/h
    dh, dw = round_half_even(h * fy), round_half_even(w * fx)
    if dw > out_w:
        raise ValueError(f"LQ width {dw} exceeds {out_w}: crop the line into shorter segments (test_sr.py:107-109)")
    lq = torch.empty((1, cn, out_h, out_w), dtype=torch.float32, device=img_u8.device)
    small = torch.empty((dh, dw, cn), dtype=torch.uint8, device=img_u8.device) if return_resized else None
    _lib.check(_lib.load().mn_preprocess_lq_u8(_ptr(img_u8), h, w, cn, fx, fy, dh, dw, _ptr(lq), _ptr(small), out_h, out_w, _stream()),
               "mn_preprocess_lq_u8")
    LAUNCHES += 1
    return (lq, dw, small) if return_resized else (lq, dw)


def postprocess_sr(sr):
    """test_sr.py:198-201 (+ cv2.imwrite's rounding): fp32 [B, C, H, W] (any strides) -> uint8 [B, H, W, C], channels flipped."""
    global LAUNCHES
    _require_cuda(sr, "sr")
    if sr.dtype != torch.float32 or sr.dim() != 4:
        raise RuntimeError("postprocess_sr: expects an fp32 [B, C, H, W] tensor")
    b, c, h, w = sr.shape
    out = torch.empty((b, h, w, c), dtype=torch.uint8, device=sr.device)
    sn, sc, sh, sw = sr.stride()
    _lib.check(_lib.load().mn_postprocess_sr_u8(_ptr(sr), sn, sc, sh, sw, _ptr(out), b, c, h, w, _stream()), "mn_postprocess_sr_u8")
    LAUNCHES += 1
    return out

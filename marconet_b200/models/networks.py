"""Host-side mirror of the reference's ``models/networks.py`` module API, executed by the
sm_100a kernels of libmarconet_b200.so through the C ABI (marconet_b200.ops).

Contract (SURVEY.md section 8b): same class names, constructor defaults, ``forward`` signatures,
return structures and ``state_dict`` keys/shapes as the reference, so the reference's
``test_sr.py`` / ``test_w.py`` run unmodified with this package providing ``models``.

Design (not a port): the nn.Module tree below only *holds parameters* under the reference's
key names.  On first use on a CUDA device the parameters are packed once
(spectral-norm sigma folded, EqualLinear scales folded, 3x3 weights re-laid K-major
``[ky,kx,Cin][Cout]``, sum-of-squares tables for demodulation, the 17 modulation FCs fused
into one GEMM) and the forward is a fixed sequence of NHWC kernels:
  - ModulatedConv2d (reference: per-sample weights + grouped conv, networks.py:281-302) is
    evaluated with ONE shared weight for all characters:
        y[n,o] = demod[n,o] * sum_k W[o,k] * (s[n,c(k)] * x[n,k])
    the style multiply is fused into the producer of x (SelectText / up-sampler / previous
    conv epilogue), demod + both biases + leaky-relu*sqrt(2) into the conv epilogue;
  - the per-character Python loops of TSPSRNet.forward (networks.py:425-448, 459-481) run as
    one ragged batch over all characters of all lines with masked windows.
There is no CPU / PyTorch fallback: inputs must live on a CUDA device.
"""
import math

import torch
import torch.nn as nn

from .. import ops
from ..ops import ACT_LRELU02, ACT_NONE, ACT_TANH
from .resnet import resnet45stride
from .textvit_arch import TextViT

SQRT2 = math.sqrt(2.0)


class _CapturedCall:
    """One module forward for one input signature, recorded into a CUDA graph: static inputs, a device error flag, static outputs."""
    __slots__ = ("graph", "inputs", "outputs", "flag", "pinned", "h2d_done")


def _copy_sources(ent, sources):
    """Caller tensors -> static inputs.  A pageable host tensor (the reference's CPU labels) would make ``copy_`` synchronise
    the stream -- the host then waits for everything queued before it (e.g. the encoder's graph) and the GPU idles while Python
    catches up -- so it is staged through a pinned buffer owned by the captured call; the event keeps the buffer from being
    overwritten while a previous copy out of it is still in flight."""
    staged = False
    for i, (st, src) in enumerate(zip(ent.inputs, sources)):
        if src.is_cuda or src.is_pinned():
            st.copy_(src, non_blocking=True)
            continue
        if ent.pinned is None:
            ent.pinned = {}
        pin = ent.pinned.get(i)
        if pin is None or pin.shape != src.shape or pin.dtype != src.dtype:
            pin = ent.pinned[i] = torch.empty(tuple(src.shape), dtype=src.dtype, pin_memory=True)
        if ent.h2d_done is not None:
            ent.h2d_done.synchronize()
        pin.copy_(src)
        st.copy_(pin, non_blocking=True)
        staged = True
    if staged:
        ent.h2d_done = torch.cuda.Event()
        ent.h2d_done.record()


class _PackedModule(nn.Module):
    """Parameter container whose packed (kernel-layout) weights are rebuilt lazily.

    Module-level CUDA graphs (round 2): the reference-facing ``forward()`` of each of the three modules is ~40-110 kernel launches
    issued from Python; the eager path paid ~1 ms of host overhead per 16-character line (launch gaps plus a GPU pipeline drain at
    every host round trip).  The SECOND call with the same input signature (shapes, device, precision plan) records the forward --
    in the same no-host-round-trip mode GraphedLines uses -- and later calls replay it: inputs are copied into static buffers,
    outputs are CLONED out of the graph's buffers (so results never alias a later call, as with the reference modules), and the
    device-side error flag is read back where the eager path would have raised.  ``MN_MODULE_GRAPHS=0`` turns it off."""

    _MG_LIMIT = 6           # captured signatures kept per module (least recently used is dropped)

    def __init__(self):
        super().__init__()
        self._packed = None
        self._packed_key = None
        self._mg = None         # OrderedDict key -> _CapturedCall | "eager"
        self._mg_hits = {}
        self.register_load_state_dict_post_hook(lambda module, incompatible: module._invalidate())

    def _invalidate(self):
        self._packed = None
        self._packed_key = None
        self._mg = None
        self._mg_hits = {}

    def _mg_run(self, key, sources, fn, fill=None):
        """Replay (or, on the second sighting of ``key``, record) ``fn(*static_inputs) -> tuple of tensors``.  ``sources`` are the
        caller's tensors (device or host) that are copied into the static inputs -- or, with ``fill``, (shape, dtype) specs of the
        static inputs, which ``fill(static_inputs)`` then writes.  Returns the captured call (static outputs, flag) or None when
        this call must run eagerly."""
        if not ops.graphs_allowed():
            return None
        import collections
        if self._mg is None:
            self._mg = collections.OrderedDict()
        key = (key, ops.graph_key())
        ent = self._mg.get(key)
        if ent is None:
            if len(self._mg_hits) > 64:
                self._mg_hits.clear()
            n = self._mg_hits.get(key, 0) + 1
            self._mg_hits[key] = n
            if n < 2:
                return None
            ent = self._mg_capture(sources, fn, fill)
            self._mg[key] = ent
            self._mg_hits.pop(key, None)
            while len(self._mg) > self._MG_LIMIT:
                self._mg.popitem(last=False)
        else:
            self._mg.move_to_end(key)
        if ent == "eager":
            return None
        if fill is not None:
            fill(ent.inputs)
        else:
            _copy_sources(ent, sources)
        ent.graph.replay()
        return ent

    def _mg_side(self, device):
        """(second stream, split-K scratch) for the parallel branch of a recorded forward; one per module."""
        side = getattr(self, "_mg_side_res", None)
        if side is None or side[1].device != device:
            side = (torch.cuda.Stream(device=device), torch.empty(ops._WS_BYTES // 4, dtype=torch.float32, device=device))
            self._mg_side_res = side
        return side

    def _mg_capture(self, sources, fn, fill):
        dev = next(self.parameters()).device
        try:
            ent = _CapturedCall()
            ent.pinned = ent.h2d_done = None
            if fill is not None:
                ent.inputs = [torch.empty(tuple(shape), dtype=dtype, device=dev) for shape, dtype in sources]
                fill(ent.inputs)
            else:
                ent.inputs = [torch.empty(tuple(s.shape), dtype=s.dtype, device=dev) for s in sources]
                _copy_sources(ent, sources)
            ent.flag = torch.zeros((1,), dtype=torch.int32, device=dev)
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side), torch.no_grad(), ops.deferred_checks(ent.flag):
                fn(*ent.inputs)                   # warm-up in the no-host-round-trip mode: fills its caches outside the capture
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            ent.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(ent.graph, capture_error_mode="thread_local"), torch.no_grad(), ops.deferred_checks(ent.flag):
                ent.flag.zero_()
                ent.outputs = tuple(fn(*ent.inputs))
            return ent
        except Exception as exc:                  # capture is an optimisation: keep the eager path for this signature
            import warnings
            warnings.warn(f"marconet_b200: CUDA-graph capture of {type(self).__name__} failed ({type(exc).__name__}: {exc}); "
                          f"this input signature keeps running eagerly")
            return "eager"

    def _apply(self, fn, *a, **k):
        self._invalidate()
        return super()._apply(fn, *a, **k)

    def _get_packed(self, device):
        first = next(self.parameters())
        if first.device != device:
            raise RuntimeError(f"marconet_b200: module parameters live on {first.device} but the input is on {device}; "
                               f"call .to(device) first (test_sr.py:66-68 does)")
        ops.poll_range(device)      # a previous call that overflowed the fp16 split re-routes its layer before we launch again
        key = (device, tuple(p._version for p in self.parameters()))
        if self._packed is None or self._packed_key != key:
            with torch.no_grad():
                self._packed = self._pack(device)
                self._pack_tc_planes(self._packed)
            self._packed_key = key
            self._mg, self._mg_hits = None, {}          # captured graphs hold the old packed weights
        return self._packed

    @staticmethod
    def _pack_tc_planes(packed):
        """Split the tensor-core layers' weights into their hi/lo 16-bit planes NOW, on the packing stream (ADVICE r1: a lazy first
        touch would run the pack kernels on whichever stream -- or graph capture -- happens to use the layer first)."""
        prec = ops.default_precision()
        if prec == ops.PREC_FP32_SIMT:
            return

        def walk(o):
            if isinstance(o, ops.ConvWeight):
                p = o.precision if o.precision is not None else prec
                if o.tc_capable() and p != ops.PREC_FP32_SIMT:
                    o.tc(p)
            elif isinstance(o, dict):
                for v in o.values():
                    walk(v)
            elif isinstance(o, (list, tuple)):
                for v in o:
                    walk(v)

        walk(packed)

    @staticmethod
    def _need_cuda(t, what):
        if not t.is_cuda:
            raise RuntimeError(f"marconet_b200.{what}: input is on {t.device}; this implementation runs only on "
                               f"CUDA (sm_100a) devices and has no CPU fallback")


def _pack_conv_weight(w, name=None):
    """[Cout, Cin, KH, KW] -> ops.ConvWeight (K-major [KH*KW*Cin, Cout] fp32 + lazily split 16-bit planes)."""
    cout, cin, kh, kw = w.shape
    return ops.ConvWeight(w.permute(2, 3, 1, 0).reshape(kh * kw * cin, cout).contiguous(), kh * kw, name=name)


# =========================================================================================
# 1) TextContextEncoderV2  (reference models/networks.py:27-45)
# =========================================================================================
class TextContextEncoderV2(_PackedModule):
    """LR line -> (char logits [B,64,6736], boxes [B,32], font style w [B,512])."""

    def __init__(self, dim=512, num_classes=6736):
        super().__init__()
        self.resnet = resnet45stride()
        self.transformer = TextViT(num_classes=num_classes, dim=512, max_length=16)

    def _pack(self, device):
        return dict(resnet=self.resnet.pack("encoder.resnet"), vit=self.transformer.pack("encoder.transformer"))

    @torch.no_grad()
    def forward(self, lq, _branch=None):
        """``_branch`` (stream, scratch): see TextViT.run -- logits / locs are produced on that stream and the caller joins it."""
        self._need_cuda(lq, "TextContextEncoderV2")
        with ops.on_device(lq):
            pk = self._get_packed(lq.device)

            def run(lq_, branch=_branch):
                x = ops.nchw_to_nhwc(lq_.float())
                feat = self.resnet.run(pk["resnet"], x)
                return self.transformer.run(pk["vit"], feat, branch=branch)

            def run_two_streams(lq_):
                # inside the recorded graph the classification / box branches run beside the style branch on a second stream
                # (own split-K scratch) and are joined before the graph ends
                br = self._mg_side(lq_.device)
                out = run(lq_, br)
                torch.cuda.current_stream(lq_.device).wait_stream(br[0])
                return out

            if _branch is None and lq.dim() == 4:
                ent = self._mg_run(("enc", tuple(lq.shape), lq.dtype, lq.device), [lq], run_two_streams)
                if ent is not None:
                    return tuple(o.clone() for o in ent.outputs)
            return run(lq)


# =========================================================================================
# 2) TSPGAN  (reference models/networks.py:51-321)
# =========================================================================================
class PixelNorm(nn.Module):
    def forward(self, input):
        return ops.pixelnorm(input)


class EqualLinear(nn.Module):
    """Parameter holder for the equalised-lr linear layer (reference networks.py:173-198)."""

    def __init__(self, in_channels, out_channels, bias=True, bias_init_val=0, lr_mul=1, activation=None):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.lr_mul, self.activation = lr_mul, activation
        self.scale = (1 / math.sqrt(in_channels)) * lr_mul
        self.weight = nn.Parameter(torch.randn(out_channels, in_channels).div_(lr_mul))
        if bias:
            self.bias = nn.Parameter(torch.zeros(out_channels).fill_(bias_init_val))
        else:
            self.register_parameter("bias", None)

    def packed(self):
        """([in, out] weight with the equalised-lr scale folded, bias * lr_mul)."""
        w = (self.weight * self.scale).t().contiguous()
        b = None if self.bias is None else (self.bias * self.lr_mul).contiguous()
        return w, b

    @torch.no_grad()
    def forward(self, x):
        w, b = self.packed()
        if self.activation == "fused_lrelu":
            return ops.linear(x.contiguous(), w, b, act=ACT_LRELU02, gain=SQRT2)
        return ops.linear(x.contiguous(), w, b)


class SelectText(nn.Module):
    def __init__(self, class_num, channel, size=4):
        super().__init__()
        self.size = size
        self.TextEmbeddings = nn.Parameter(torch.randn(class_num, channel, 1, 1))


class FusedLeakyReLU(nn.Module):
    """Holds the ``activate.bias`` parameter of the third-party basicsr FusedLeakyReLU."""

    def __init__(self, channel):
        super().__init__()
        self.bias = nn.Parameter(torch.zeros(channel))


class ModulatedConv2d(nn.Module):
    def __init__(self, in_channel, out_channel, kernel_size, style_dim, demodulate=True, upsample=False,
                 downsample=False, blur_kernel=[1, 3, 3, 1]):
        super().__init__()
        self.eps = 1e-8
        self.kernel_size, self.in_channel, self.out_channel = kernel_size, in_channel, out_channel
        self.upsample, self.downsample, self.demodulate = upsample, downsample, demodulate
        self.scale = 1 / math.sqrt(in_channel * kernel_size ** 2)
        self.padding = kernel_size // 2
        self.weight = nn.Parameter(torch.randn(1, out_channel, in_channel, kernel_size, kernel_size))
        self.modulation = EqualLinear(style_dim, in_channel, bias=True, bias_init_val=1, lr_mul=1, activation=None)


class StyledConv(nn.Module):
    def __init__(self, in_channel, out_channel, kernel_size, style_dim, upsample=False, blur_kernel=[1, 3, 3, 1],
                 demodulate=True):
        super().__init__()
        self.conv = ModulatedConv2d(in_channel, out_channel, kernel_size, style_dim, upsample=upsample,
                                    blur_kernel=blur_kernel, demodulate=demodulate)
        self.bias = nn.Parameter(torch.zeros(1, out_channel, 1, 1))
        self.activate = FusedLeakyReLU(out_channel)


class ToRGB(nn.Module):
    def __init__(self, in_channel, style_dim, upsample=True, blur_kernel=[1, 3, 3, 1]):
        super().__init__()
        self.upsample = upsample
        self.conv = ModulatedConv2d(in_channel, 3, 1, style_dim, demodulate=False)
        self.bias = nn.Parameter(torch.zeros(1, 3, 1, 1))


class TextGenerator(_PackedModule):
    """font style w + character labels -> (128-px structure image, 64x64 prior, 32x32 prior)."""

    def __init__(self, size, style_dim, n_mlp, class_num, channel_multiplier=1, blur_kernel=[1, 3, 3, 1], lr_mlp=0.01):
        super().__init__()
        self.size, self.n_mlp, self.style_dim = size, n_mlp, style_dim
        self.style_mlp = nn.Sequential(PixelNorm(), *[
            EqualLinear(style_dim, style_dim, bias=True, bias_init_val=0, lr_mul=lr_mlp, activation="fused_lrelu")
            for _ in range(n_mlp)])
        m = channel_multiplier
        self.channels = {4: 512, 8: 512, 16: 512, 32: 512, 64: 256 * m, 128: 128 * m, 256: 64 * m, 512: 32 * m, 1024: 16 * m}
        self.input_text = SelectText(class_num, self.channels[4])
        self.conv1 = StyledConv(self.channels[4], self.channels[4], 3, style_dim, blur_kernel=blur_kernel)
        self.to_rgb1 = ToRGB(self.channels[4], style_dim, upsample=False)
        self.log_size = int(math.log(size, 2))
        self.convs, self.upsamples, self.to_rgbs = nn.ModuleList(), nn.ModuleList(), nn.ModuleList()
        cin = self.channels[4]
        for i in range(3, self.log_size + 1):
            cout = self.channels[2 ** i]
            self.convs.append(StyledConv(cin, cout, 3, style_dim, upsample=True, blur_kernel=blur_kernel))
            self.convs.append(StyledConv(cout, cout, 3, style_dim, blur_kernel=blur_kernel))
            self.to_rgbs.append(ToRGB(cout, style_dim))
            cin = cout
        self.n_latent = self.log_size * 2 - 2

    # ---- pack -----------------------------------------------------------------------------
    def _pack(self, device):
        pk = {}
        pk["mlp"] = [m.packed() for m in list(self.style_mlp)[1:]]
        styled = [self.conv1] + list(self.convs)
        rgbs = [self.to_rgb1] + list(self.to_rgbs)
        # one GEMM for all 17 modulation FCs: columns [conv1 | convs.* | to_rgb1 | to_rgbs.*]
        mods = [m.conv.modulation for m in styled] + [m.conv.modulation for m in rgbs]
        ws, bs, offs, off = [], [], [], 0
        for mod in mods:
            w, b = mod.packed()
            ws.append(w); bs.append(b); offs.append((off, w.shape[1])); off += w.shape[1]
        pk["mod_w"] = torch.cat(ws, dim=1).contiguous()
        pk["mod_b"] = torch.cat(bs).contiguous()
        pk["mod_total"] = off
        pk["styled"] = []
        for i, m in enumerate(styled):
            w = m.conv.weight[0] * m.conv.scale                      # [Cout, Cin, 3, 3]  (networks.py:284)
            pk["styled"].append(dict(
                w=_pack_conv_weight(w, "tspgan." + ("conv1" if i == 0 else f"convs.{i - 1}")), wsq=w.pow(2).sum([2, 3]).t().contiguous(),   # [Cin, Cout]
                bias=(m.bias.reshape(-1) + m.activate.bias).contiguous(),
                off=offs[i], up=m.conv.upsample, cout=w.shape[0]))
        pk["rgb"] = []
        for i, m in enumerate(rgbs):
            w = (m.conv.weight[0, :, :, 0, 0] * m.conv.scale).contiguous()          # [3, Cin]
            pk["rgb"].append(dict(w=w, bias=m.bias.reshape(-1).contiguous(), off=offs[len(styled) + i]))
        pk["emb"] = self.input_text.TextEmbeddings[:, :, 0, 0].contiguous()
        entries, off = [], 0
        for e in pk["styled"]:
            entries.append((e["wsq"], e["off"][0], off))
            e["demod_off"] = off
            off += e["cout"]
        pk["demod_table"] = ops.make_demod_table(entries, device)
        pk["demod_total"] = off
        return pk

    # ---- forward --------------------------------------------------------------------------
    @torch.no_grad()
    def forward(self, styles, labels, noise=None, _branch=None, _tap_ptrs=None):
        """``_branch``: a second CUDA stream for the ToRGB chain (the 128-px prior image), which the feature taps -- and hence the
        SR decoder -- do not depend on; the CALLER joins that stream before it reads the image.
        ``_tap_ptrs`` = {64: ptrs, 32: ptrs} (int64 device tensors, one destination address per character): the two feature taps
        are ADDITIONALLY stored through these per-character pointers by the epilogue of the convolution that produces them
        (mn_conv_params.y2_ptrs) -- marconet_b200.parallel.PeerPriorExchange points them into the symmetric-memory buffers of
        the ranks that own the characters' lines."""
        self._need_cuda(styles, "TSPGAN")
        with ops.on_device(styles):
            if _tap_ptrs is not None:
                return self._forward(styles, labels, _branch, _tap_ptrs)
            if _branch is None and labels.dim() == 2 and styles.dim() == 2 and styles.shape[0] == labels.shape[0] and labels.numel() > 0:
                self._get_packed(styles.device)
                classes = self.input_text.TextEmbeddings.shape[0]
                if not labels.is_cuda:      # the reference's caller keeps labels on the CPU (test_sr.py:180): host check, no round trip
                    lab64 = labels.detach().to(torch.int64)
                    if int(lab64.min()) < 0 or int(lab64.max()) >= classes:
                        raise IndexError(f"character label out of range [0, {classes}) (reference: empty embedding slice, networks.py:211)")
                else:
                    lab64 = labels.detach().to(torch.int64)
                def run_two_streams(st_, lab_):
                    # inside the recorded graph the ToRGB chain (the prior image) runs on a second stream beside the main convs
                    br = self._mg_side(st_.device)[0]
                    out = self._forward(st_, lab_, br)
                    torch.cuda.current_stream(st_.device).wait_stream(br)
                    return out

                ent = self._mg_run(("gen", tuple(styles.shape), tuple(labels.shape), styles.dtype, styles.device), [styles, lab64],
                                   run_two_streams)
                if ent is not None:
                    if labels.is_cuda:      # device-side range check: read the flag where the eager path would have raised
                        ops.raise_deferred(int(ent.flag.item()))
                    return tuple(o.clone() for o in ent.outputs)
            return self._forward(styles, labels, _branch)

    def _forward(self, styles, labels, _branch, _tap_ptrs=None):
        dev = styles.device
        pk = self._get_packed(dev)
        if labels.dim() != 2:
            raise RuntimeError("labels must be [N, L]")
        n, l = labels.shape
        if styles.shape[0] != n:
            raise RuntimeError("styles and labels disagree on the number of characters")
        flag = ops.deferred_flag()
        if flag is not None and labels.is_cuda:
            # no host round trip (CUDA-graph capture): range check + clamp on the device, error bit read back by the caller
            lab_dev = ops.check_labels(labels.to(torch.int64).contiguous().reshape(-1), pk["emb"].shape[0], flag)
        else:
            lab_host = labels.detach().to("cpu", torch.int64)
            if n * l > 0 and (int(lab_host.min()) < 0 or int(lab_host.max()) >= pk["emb"].shape[0]):
                raise IndexError(f"character label out of range [0, {pk['emb'].shape[0]}) "
                                 f"(reference: empty embedding slice, networks.py:211)")
            lab_dev = labels.to(dev, torch.int64).contiguous().reshape(-1) if labels.is_cuda else \
                lab_host.reshape(-1).to(dev, non_blocking=False)

        z = ops.pixelnorm(styles.float().contiguous())
        for w, b in pk["mlp"]:
            z = ops.linear(z, w, b, act=ACT_LRELU02, gain=SQRT2)
        s_all = ops.linear(z, pk["mod_w"], pk["mod_b"])              # [N, 7168]

        def s_of(entry):
            o, c = entry["off"]
            return s_all[:, o:o + c]

        st = pk["styled"]
        demod_all = ops.demod_batched(s_all, pk["demod_table"], pk["demod_total"])       # [N, sum Cout], one launch
        demods = [demod_all[:, e["demod_off"]:e["demod_off"] + e["cout"]] for e in st]

        def styled(i, x, want_y, next_i=None, tap_ptrs=None):
            e = st[i]
            y2s = None if next_i is None else s_of(st[next_i])
            return ops.conv2d(x, e["w"], 3, 3, pad=(1, 1), bias=e["bias"], out_scale=demods[i], act=ACT_LRELU02,
                              gain=SQRT2, want_y=want_y, out2=(True if next_i is not None else None), y2_scale=y2s, out2_ptrs=tap_ptrs)

        main = torch.cuda.current_stream(dev) if _branch is not None else None

        def rgb(y, r, skip):
            if _branch is None:
                return ops.torgb(y, s_of(r), r["w"], r["bias"], skip)
            _branch.wait_stream(main)                               # y (and s_all) are ready on the main stream
            y.record_stream(_branch)
            s_all.record_stream(_branch)                            # the style slices are read on the branch after forward() returns
            with torch.cuda.stream(_branch):
                out = ops.torgb(y, s_of(r), r["w"], r["bias"], skip)
            out.record_stream(main)
            return out

        x = ops.select_text(pk["emb"], lab_dev, s_of(st[0]), n, l)   # embedding * style(conv1)
        y = styled(0, x, True)
        skip = rgb(y, pk["rgb"][0], None)
        taps = {}
        for j in range(len(self.to_rgbs)):
            ia, ib = 1 + 2 * j, 2 + 2 * j
            xu = ops.resample_modulate(y, s_of(st[ia]), up=True)     # bilinear x2 of the un-modulated map, then style
            xm = styled(ia, xu, False, next_i=ib)                    # only the pre-modulated operand of conv b is kept
            tp = None if (_tap_ptrs is None or l != 1) else _tap_ptrs.get(xm.shape[2])     # the tap layers (64 / 32 columns wide)
            y = styled(ib, xm, True, tap_ptrs=tp)
            skip = rgb(y, pk["rgb"][1 + j], skip)
            taps[y.shape[2]] = y                                     # the reference picks its taps by WIDTH (networks.py:153-158)
        if 64 not in taps or 32 not in taps:
            raise RuntimeError(f"labels [N, {l}]: no feature map is 64 / 32 columns wide (the reference leaves its taps unset, "
                               f"networks.py:153-158)")
        return ops.as_nchw_view(skip), ops.as_nchw_view(taps[64]), ops.as_nchw_view(taps[32])


class TSPGAN(nn.Module):
    def __init__(self, out_size=128, num_style_feat=512, class_num=6736, num_mlp=8):
        super().__init__()
        self.TextGenerator = TextGenerator(size=out_size, style_dim=num_style_feat, n_mlp=num_mlp, class_num=class_num)

    def forward(self, styles, labels, noise, _branch=None, _tap_ptrs=None):
        return self.TextGenerator(styles, labels, noise, _branch=_branch, _tap_ptrs=_tap_ptrs)


# =========================================================================================
# 3) TSPSRNet  (reference models/networks.py:328-533)
# =========================================================================================
class _SNConv(nn.Module):
    """Spectral-norm 3x3 conv parameter holder with torch.nn.utils.spectral_norm's state_dict keys
    (bias, weight_orig, weight_u, weight_v).  sigma is folded into the weight once at pack time
    (eval branch of spectral_norm: W / (u . W_mat v))."""

    def __init__(self, cin, cout, stride=1):
        super().__init__()
        self.in_channels, self.out_channels, self.stride = cin, cout, stride
        conv = nn.Conv2d(cin, cout, 3, stride, 1)
        self.bias = nn.Parameter(conv.bias.detach().clone())
        self.weight_orig = nn.Parameter(conv.weight.detach().clone())
        wm = self.weight_orig.detach().flatten(1)
        u = nn.functional.normalize(torch.randn(cout), dim=0, eps=1e-12)
        v = nn.functional.normalize(torch.randn(cin * 9), dim=0, eps=1e-12)
        for _ in range(8):   # settle sigma so that a default-initialised net is finite in eval mode
            v = nn.functional.normalize(torch.mv(wm.t(), u), dim=0, eps=1e-12)
            u = nn.functional.normalize(torch.mv(wm, v), dim=0, eps=1e-12)
        self.register_buffer("weight_u", u)
        self.register_buffer("weight_v", v)

    def packed(self, name=None):
        w = self.weight_orig
        sigma = torch.dot(self.weight_u, torch.mv(w.flatten(1), self.weight_v))
        return _pack_conv_weight(w / sigma, name), self.bias.contiguous()


class _Slot(nn.Module):
    """Parameter-free placeholder keeping nn.Sequential indices aligned with the reference
    (LeakyReLU / Upsample / Tanh positions)."""

    def __init__(self, what):
        super().__init__()
        self.what = what

    def extra_repr(self):
        return self.what


def GroupNorm(in_channels):
    assert in_channels % 32 == 0
    return nn.GroupNorm(num_groups=in_channels // 32, num_channels=in_channels, eps=1e-6, affine=True)


class ResTextBlockV2(nn.Module):
    def __init__(self, in_channels, out_channels=None):
        super().__init__()
        self.in_channels = in_channels
        self.out_channels = in_channels if out_channels is None else out_channels
        self.norm1 = GroupNorm(in_channels)
        self.conv1 = _SNConv(in_channels, self.out_channels)
        self.norm2 = GroupNorm(self.out_channels)
        self.conv2 = _SNConv(self.out_channels, self.out_channels)
        if self.in_channels != self.out_channels:
            self.conv_out = nn.Conv2d(in_channels, self.out_channels, kernel_size=1, stride=1, padding=0)

    def packed(self, name=None):
        nm = (lambda s: None) if name is None else (lambda s: f"{name}.{s}")
        d = dict(n1=(self.norm1.weight.contiguous(), self.norm1.bias.contiguous()), c1=self.conv1.packed(nm("conv1")),
                 n2=(self.norm2.weight.contiguous(), self.norm2.bias.contiguous()), c2=self.conv2.packed(nm("conv2")), co=None)
        if self.in_channels != self.out_channels:
            d["co"] = (_pack_conv_weight(self.conv_out.weight, nm("conv_out")), self.conv_out.bias.contiguous())
        return d


def _res_block(pk, x, valid_w=None, mr1=None):
    """GN -> swish -> conv -> GN -> swish -> conv (+ 1x1 skip), reference networks.py:506-516.
    ``mr1``: statistics of x when the convolution that produced x already accumulated them in its epilogue."""
    # normalise + swish is the tcgen05 kernel's operand transform (ops.FUSE_GN, default on: no separate pass over x); layers the
    # fp32 kernel runs, or MN_FUSE_GN=0, take mn_groupnorm_apply first
    if mr1 is None:
        mr1 = ops.groupnorm_stats(x, valid_w=valid_w)
    # the statistics of h (input of norm2) are accumulated by the epilogue of the conv that writes h: no separate read pass
    h, mr2 = ops.conv2d(x, pk["c1"][0], 3, 3, pad=(1, 1), bias=pk["c1"][1], valid_w=valid_w, gn=(mr1,) + tuple(pk["n1"]), gn_stats=True)
    skip = x if pk["co"] is None else ops.conv2d(x, pk["co"][0], 1, 1, bias=pk["co"][1], valid_w=valid_w)
    return ops.conv2d(h, pk["c2"][0], 3, 3, pad=(1, 1), bias=pk["c2"][1], residual=skip, valid_w=valid_w, gn=(mr2,) + tuple(pk["n2"]))


def _two(pk, x, valid_w=None):
    """SN-conv -> LeakyReLU(0.2) -> SN-conv."""
    t = ops.conv2d(x, pk[0][0], 3, 3, pad=(1, 1), bias=pk[0][1], act=ACT_LRELU02, valid_w=valid_w)
    return ops.conv2d(t, pk[1][0], 3, 3, pad=(1, 1), bias=pk[1][1], valid_w=valid_w)


def _char_windows_np(arr, counts, width, half):
    """Vectorised core of char_windows.  ``arr``: fp32 numpy [B, >= 2*n].  The centre is the fp32 product truncated toward zero,
    exactly like ``(locs[b][2*c] * W).int()`` (numpy float32 array x np.float32 scalar is an fp32 multiply; astype(int32) truncates).
    Returns (wins int32 [Nc,4] = (line, x1, x2, y1), valid int32 [Nc], owner int32 [B, W])."""
    import numpy as np
    nc = sum(counts)
    wins = np.empty((nc, 4), np.int32)
    valid = np.empty((nc,), np.int32)
    owner = np.full((len(counts), width), -1, np.int32)
    w32 = np.float32(width)
    i = 0
    for b, n in enumerate(counts):
        if n == 0:
            continue
        cen = (arr[b, 0:2 * n:2].astype(np.float32, copy=False) * w32).astype(np.int32)
        x1 = np.where(cen < half, 0, cen - half)
        x2 = np.where(cen + half > width, width, cen + half)
        wv = x2 - x1
        bad = np.nonzero((wv <= 0) | (x1 >= width))[0]
        if bad.size:
            c = int(bad[0])
            raise RuntimeError(f"character {c} of line {b}: empty window (centre {int(cen[c])}); the reference "
                               f"fails on the empty slice at networks.py:443")
        wins[i:i + n, 0] = b
        wins[i:i + n, 1] = x1
        wins[i:i + n, 2] = x2
        wins[i:i + n, 3] = half - wv // 2            # wv > 0: floor division == the reference's trunc division
        valid[i:i + n] = wv
        for c in range(n):                           # program order: the last writer wins (networks.py:448,481)
            owner[b, x1[c]:x2[c]] = i + c
        i += n
    return wins, valid, owner


def char_windows(locs_host, counts, width, half):
    """Bit-exact restatement of the window integers of reference networks.py:426-441 / :460-474.

    ``locs_host`` is a CPU fp32 tensor [B, 2*n]; the centre is ``(locs[b][2c] * W).int()`` (fp32
    multiply, truncation).  Returns (windows [(line,x1,x2,y1)], valid widths, owner[b][x]) with
    "last character in program order wins" ownership (networks.py:448,481).
    """
    wins, valid, owner = _char_windows_np(locs_host.detach().to(torch.float32).contiguous().numpy(), counts, width, half)
    return [tuple(int(v) for v in r) for r in wins], [int(v) for v in valid], owner.tolist()


class TSPSRNet(_PackedModule):
    """LR line + per-character structure priors + boxes -> SR line [B,3,128,2048]."""

    def __init__(self, in_channel=3, dim_channel=256):
        super().__init__()
        d = dim_channel
        act, up = (lambda: _Slot("LeakyReLU(0.2)")), (lambda: _Slot("Upsample(x2, bilinear)"))
        self.conv_first_32 = nn.Sequential(_SNConv(in_channel, d // 4), act())
        self.conv_first_16 = nn.Sequential(_SNConv(d // 4, d // 2, 2), act())
        self.conv_first_8 = nn.Sequential(_SNConv(d // 2, d, 2), act(), _SNConv(d, d))
        self.conv_body_16 = nn.Sequential(_SNConv(d + d // 2, d), act(), _SNConv(d, d))
        self.conv_body_32 = nn.Sequential(_SNConv(d + d // 4, d), act(), _SNConv(d, d))
        self.conv_up = nn.Sequential(up(), _SNConv(d, d), act(), ResTextBlockV2(d, d), _SNConv(d, d))
        self.conv_final = nn.Sequential(_SNConv(d, d // 2), act(), up(), _SNConv(d // 2, d // 4), act(),
                                        ResTextBlockV2(d // 4, d // 4), _SNConv(d // 4, 3), _Slot("Tanh"))
        self.conv_32_scale = nn.Sequential(_SNConv(d, d), act(), _SNConv(d, d))
        self.conv_32_shift = nn.Sequential(_SNConv(d, d), act(), _SNConv(d, d))
        self.conv_32_fuse = nn.Sequential(ResTextBlockV2(2 * d, d))
        self.conv_32_to256 = nn.Sequential(_SNConv(512, d), act(), _SNConv(d, d))
        self.conv_64_scale = nn.Sequential(_SNConv(d, d), act(), _SNConv(d, d))
        self.conv_64_shift = nn.Sequential(_SNConv(d, d), act(), _SNConv(d, d))
        self.conv_64_fuse = nn.Sequential(ResTextBlockV2(2 * d, d))
        self.dim = d
        self._line_first_cache = {}

    def _pack(self, device):
        pk = {}
        for name in ("conv_first_8", "conv_body_16", "conv_body_32", "conv_32_scale", "conv_32_shift", "conv_32_to256",
                     "conv_64_scale", "conv_64_shift"):
            seq = getattr(self, name)
            pk[name] = (seq[0].packed(f"sr.{name}.0"), seq[2].packed(f"sr.{name}.2"))
        pk["first_32"] = self.conv_first_32[0].packed("sr.conv_first_32.0")
        pk["first_16"] = self.conv_first_16[0].packed("sr.conv_first_16.0")
        pk["up_1"] = self.conv_up[1].packed("sr.conv_up.1")
        pk["up_res"] = self.conv_up[3].packed("sr.conv_up.3")
        pk["up_4"] = self.conv_up[4].packed("sr.conv_up.4")
        pk["fin_0"] = self.conv_final[0].packed("sr.conv_final.0")
        pk["fin_3"] = self.conv_final[3].packed("sr.conv_final.3")
        pk["fin_res"] = self.conv_final[5].packed("sr.conv_final.5")
        pk["fin_6"] = self.conv_final[6].packed("sr.conv_final.6")
        pk["fuse32"] = self.conv_32_fuse[0].packed("sr.conv_32_fuse.0")
        pk["fuse64"] = self.conv_64_fuse[0].packed("sr.conv_64_fuse.0")
        return pk

    def _line_first(self, counts, dev):
        """Device int32[B+1] prefix sums of the per-line character counts (cached: constant for a captured graph)."""
        key = (tuple(counts), dev)
        t = self._line_first_cache.get(key)
        if t is None:
            pre = [0]
            for n in counts:
                pre.append(pre[-1] + n)
            t = torch.tensor(pre, dtype=torch.int32).to(dev)
            self._line_first_cache[key] = t
        return t

    def _fuse(self, pk, lvl, feat, prior, locs, counts, half):
        """Per-character prior fusion of one level as ONE ragged batch (reference loops :425-448/:459-481).
        ``locs`` is a CPU tensor (eager checks) or, inside ops.deferred_checks, the device tensor itself."""
        dev = feat.device
        b, h, w, c = feat.shape
        nc = sum(counts)
        if nc == 0:
            return feat
        wp = 2 * half
        flag = ops.deferred_flag()
        if flag is not None and locs.is_cuda:
            win_dev, valid_dev, owner_dev = ops.char_windows(locs, self._line_first(counts, dev), counts, w, half, flag)
            vw = valid_dev                                # widths are not known on the host: always mask
        else:
            wins, valid, owner = _char_windows_np(locs.numpy() if isinstance(locs, torch.Tensor) else locs, counts, w, half)
            win_dev = torch.from_numpy(wins).to(dev, non_blocking=True)
            valid_dev = torch.from_numpy(valid).to(dev, non_blocking=True)
            owner_dev = torch.from_numpy(owner).to(dev, non_blocking=True)
            vw = valid_dev if int(valid.min()) < wp else None   # full-width windows need no masking
        fin = ops.adain_concat(prior, feat, win_dev, nc, wp)                         # [Nc,H,wp,2C]
        fuse = _res_block(pk[f"fuse{lvl}"], fin, vw)
        scale = _two(pk[f"conv_{lvl}_scale"], fuse, vw)
        shift = _two(pk[f"conv_{lvl}_shift"], fuse, vw)
        return ops.window_scatter(feat, scale, shift, owner_dev, win_dev, wp)

    @staticmethod
    def _gather_priors(priors, channels, size):
        views = []
        for p in priors:
            if p.dim() != 4 or p.shape[1] != channels or p.shape[2] != size or p.shape[3] != size:
                raise RuntimeError(f"prior has shape {tuple(p.shape)}, expected [n,{channels},{size},{size}]")
            views.append(ops.as_nhwc(p.float()))
        if len(views) == 1:
            return views[0]
        # priors of consecutive lines that are slices of ONE generator call are already adjacent in memory: re-join them
        # without a copy; anything else is concatenated.
        nxt, total = views[0].data_ptr(), 0
        for v in views:
            if not v.is_contiguous() or v.data_ptr() != nxt or v.untyped_storage().data_ptr() != views[0].untyped_storage().data_ptr():
                return torch.cat(views, dim=0)
            nxt += v.numel() * 4
            total += v.shape[0]
        return torch.as_strided(views[0], (total,) + tuple(views[0].shape[1:]), views[0].stride())

    def _trunk(self, pk, lq):
        """The LR trunk (reference networks.py:412-416): depends on the LR line only, not on the priors."""
        dev, d = lq.device, self.dim
        bsz = lq.shape[0]
        x = ops.nchw_to_nhwc(lq.float())
        h, w = x.shape[1], x.shape[2]
        cat32 = torch.empty((bsz, h, w, d + d // 4), dtype=torch.float32, device=dev)        # [up(sq_f_16) | lq_f_32]
        cat16 = torch.empty((bsz, h // 2, w // 2, d + d // 2), dtype=torch.float32, device=dev)  # [up(lq_f_8) | lq_f_16]
        f32v, f16v = cat32[..., d:], cat16[..., d:]
        ops.conv2d(x, pk["first_32"][0], 3, 3, pad=(1, 1), bias=pk["first_32"][1], act=ACT_LRELU02, out=f32v)
        ops.conv2d(f32v, pk["first_16"][0], 3, 3, stride=(2, 2), pad=(1, 1), bias=pk["first_16"][1], act=ACT_LRELU02, out=f16v)
        p8 = pk["conv_first_8"]
        t = ops.conv2d(f16v, p8[0][0], 3, 3, stride=(2, 2), pad=(1, 1), bias=p8[0][1], act=ACT_LRELU02)
        f8 = ops.conv2d(t, p8[1][0], 3, 3, pad=(1, 1), bias=p8[1][1])
        ops.resample_modulate(f8, None, up=True, out=cat16[..., :d])
        s16 = _two(pk["conv_body_16"], cat16)
        ops.resample_modulate(s16, None, up=True, out=cat32[..., :d])
        s32 = _two(pk["conv_body_32"], cat32)
        return s32

    @staticmethod
    def _check_geometry(lq, priors32=()):
        """Shapes the reference module rejects, raised before anything is launched: the two stride-2 convs and the two x2
        up-samplings of the trunk only line up (torch.cat at networks.py:415-416) when H and W are multiples of 4, and the 32-px
        priors are concatenated with H-row windows of the 32-level map (networks.py:442-445), so H must be 32 when any line has
        characters.  (Without the first check, W = 2 mod 4 would make the up-sampled 8-row map one column wider than its slot.)"""
        if lq.dim() != 4:
            raise RuntimeError(f"TSPSRNet: lq must be [B, 3, H, W], got {tuple(lq.shape)}")
        h, w = int(lq.shape[2]), int(lq.shape[3])
        if h % 4 or w % 4:
            raise RuntimeError(f"TSPSRNet: LR line of {h}x{w}; height and width must be multiples of 4 (the reference fails in "
                               f"torch.cat at networks.py:415-416)")
        if h != 32 and any(int(p.shape[0]) > 0 for p in priors32):
            raise RuntimeError(f"TSPSRNet: LR line height {h} with characters; the 32x32 priors need height 32 (networks.py:442-445)")

    @torch.no_grad()
    def trunk(self, lq):
        """Public handle on the LR trunk so that a pipeline can launch it early, on a second stream, while the encoder and the
        prior generator run (it needs only the LR line): pass the result to forward(..., _trunk=...)."""
        self._need_cuda(lq, "TSPSRNet")
        self._check_geometry(lq)
        with ops.on_device(lq):
            return self._trunk(self._get_packed(lq.device), lq)

    @torch.no_grad()
    def forward(self, lq, priors64, priors32, locs, _trunk=None):
        self._need_cuda(lq, "TSPSRNet")
        self._check_geometry(lq, priors32)
        with ops.on_device(lq):
            ent = self._forward_graphed(lq, priors64, priors32, locs) if _trunk is None else None
            if ent is not None:
                ops.raise_deferred(int(ent.flag.item()))      # the eager path raises on an empty window before launching; here after
                return ent.outputs[0].clone()
            return self._forward(lq, priors64, priors32, locs, _trunk)

    def _forward_graphed(self, lq, priors64, priors32, locs):
        """Module-level CUDA graph of the decoder for this (lines, characters-per-line) signature; None -> run eagerly."""
        if not ops.graphs_allowed() or lq.dim() != 4 or len(priors64) != len(priors32) or not isinstance(locs, torch.Tensor) or locs.dim() != 2:
            return None
        bsz = lq.shape[0]
        counts = [int(p.shape[0]) for p in priors32] + [0] * (bsz - len(priors32))
        nc = sum(counts)
        d = self.dim
        if (nc == 0 or len(priors64) != bsz or min(counts) == 0 or [int(p.shape[0]) for p in priors64] != counts
                or locs.shape[0] < bsz or locs.shape[1] < 2 * max(counts)):
            return None
        for p, ch, sz in [(p, d, 64) for p in priors64] + [(p, 512, 32) for p in priors32]:
            if p.dim() != 4 or tuple(p.shape[1:]) != (ch, sz, sz) or not p.is_cuda:
                return None
        self._get_packed(lq.device)
        # static inputs: the LR lines, the boxes, and all priors of all lines as two NHWC tensors (each line's priors are copied
        # straight into their slice: one contiguous device copy per line when the caller passes the generator's own outputs)
        specs = [(lq.shape, torch.float32), (locs.shape, torch.float32), ((nc, 64, 64, d), torch.float32), ((nc, 32, 32, 512), torch.float32)]

        def fill(st):
            st[0].copy_(lq, non_blocking=True)
            st[1].copy_(locs.detach(), non_blocking=True)
            o = 0
            for i, n in enumerate(counts[:len(priors64)]):
                if n:
                    st[2][o:o + n].copy_(priors64[i].permute(0, 2, 3, 1), non_blocking=True)
                    st[3][o:o + n].copy_(priors32[i].permute(0, 2, 3, 1), non_blocking=True)
                o += n

        def run(lq_, locs_, p64_, p32_):
            l64, l32, o = [], [], 0
            for n in counts:
                l64.append(p64_[o:o + n].permute(0, 3, 1, 2)); l32.append(p32_[o:o + n].permute(0, 3, 1, 2)); o += n
            return (self._forward(lq_, l64[:len(priors64)], l32[:len(priors32)], locs_, None, _trunk_side=self._mg_side(lq_.device)),)

        key = ("sr", tuple(lq.shape), tuple(counts), len(priors64), tuple(locs.shape), lq.device)
        return self._mg_run(key, specs, run, fill)

    def _forward(self, lq, priors64, priors32, locs, _trunk, _trunk_side=None):
        """``_trunk_side`` = (stream, split-K scratch): compute the LR trunk on that stream while this one converts the 32-px priors
        (they are independent: networks.py:412-416 vs :424); joined before the first fuse stage.  Used inside recorded graphs."""
        dev = lq.device
        pk = self._get_packed(dev)
        d = self.dim
        bsz = lq.shape[0]
        if len(priors64) != len(priors32):
            raise RuntimeError("priors64 and priors32 must have one entry per line")
        counts = [int(p.shape[0]) for p in priors32] + [0] * (bsz - len(priors32))
        if [int(p.shape[0]) for p in priors64] != counts[:len(priors64)]:
            raise RuntimeError("priors64 / priors32 disagree on the number of characters")
        if ops.deferred_flag() is not None and locs.is_cuda:
            locs_host = locs.detach().float().contiguous()      # stays on the device; windows come from mn_char_windows
        else:
            locs_host = locs.detach().to("cpu", torch.float32).contiguous()      # the one device->host round trip (reference: ~6 per character)

        trunk_done = None
        if _trunk is not None:
            s32 = _trunk
        elif _trunk_side is not None and sum(counts) > 0:
            side, scratch = _trunk_side
            main = torch.cuda.current_stream(dev)
            side.wait_stream(main)
            with torch.cuda.stream(side), ops.use_workspace(scratch):
                s32 = self._trunk(pk, lq)
                trunk_done = torch.cuda.Event()
                trunk_done.record(side)
            s32.record_stream(main)
        else:
            s32 = self._trunk(pk, lq)

        if sum(counts) > 0:
            p32 = _two(pk["conv_32_to256"], self._gather_priors(priors32, 512, 32))
            if trunk_done is not None:
                torch.cuda.current_stream(dev).wait_event(trunk_done)
            s32 = self._fuse(pk, 32, s32, p32, locs_host, counts, 16)

        u = ops.resample_modulate(s32, None, up=True)
        x, mr = ops.conv2d(u, pk["up_1"][0], 3, 3, pad=(1, 1), bias=pk["up_1"][1], act=ACT_LRELU02, gn_stats=True)
        x = _res_block(pk["up_res"], x, mr1=mr)
        s64 = ops.conv2d(x, pk["up_4"][0], 3, 3, pad=(1, 1), bias=pk["up_4"][1])

        if sum(counts) > 0:
            s64 = self._fuse(pk, 64, s64, self._gather_priors(priors64, d, 64), locs_host, counts, 32)

        x = ops.conv2d(s64, pk["fin_0"][0], 3, 3, pad=(1, 1), bias=pk["fin_0"][1], act=ACT_LRELU02)
        u = ops.resample_modulate(x, None, up=True)
        x, mr = ops.conv2d(u, pk["fin_3"][0], 3, 3, pad=(1, 1), bias=pk["fin_3"][1], act=ACT_LRELU02, gn_stats=True)
        x = _res_block(pk["fin_res"], x, mr1=mr)
        out = ops.conv2d(x, pk["fin_6"][0], 3, 3, pad=(1, 1), bias=pk["fin_6"][1], act=ACT_TANH)
        return ops.as_nchw_view(out)


def swish(x):
    """reference networks.py:492-493 (the hot path fuses it into the GroupNorm apply; this is the standalone function)."""
    with ops.on_device(x):
        return ops.swish(x.float())


def calc_mean_std_4D(feat, eps=1e-5):
    """reference networks.py:518-525."""
    with ops.on_device(feat):
        return ops.calc_mean_std_4d(feat.float(), eps)


def adaptive_instance_normalization(prior_feat, lq_feat):
    """reference networks.py:528-533 (the hot path uses the fused, window-aware mn_adain_concat)."""
    with ops.on_device(prior_feat):
        return ops.adaptive_instance_normalization(prior_feat.float(), lq_feat.float())

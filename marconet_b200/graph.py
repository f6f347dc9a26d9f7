"""CUDA-graph capture of the whole line pipeline (SURVEY.md section 8f row n1).

The reference restores one line at a time with Python loops over the characters (test_sr.py:77, networks.py:425,459) and a
device->host round trip wherever a box coordinate becomes a Python int (networks.py:426-441).  Here one step = encoder ->
TSPGAN (all characters of all lines in one call) -> TSPSRNet for a FIXED shape (``lines`` x ``chars``) is recorded once into a
CUDA graph and replayed: no Python between the ~220 launches, no host round trip (label range check and window integers run
as device kernels inside ``ops.deferred_checks``; their error bits are read back together with the result).

The flow is the one of test_sr.py: labels and boxes come from the caller (OCR / detector), the style ``w`` from the encoder.
Lines wider than 512 columns (``width`` a multiple of 64) follow pipeline.restore_wide_image: the encoder runs on the 512-column
segments of every line and each character takes the style of the segment that holds its centre (mn_char_segment_styles).
"""
import torch

from . import ops


class GraphedLines:
    """encoder -> TSPGAN -> TSPSRNet for ``lines`` LR lines of ``chars`` characters each, as one CUDA graph.

    >>> g = GraphedLines(encoder, tspgan, sr, lines=1, chars=16)
    >>> out = g(lq, labels, locs)      # lq [lines,3,32,width] fp32, labels int64 [lines*chars,1], locs fp32 [lines,2*chars]
    >>> g.check()                      # raises what the eager modules would have raised (reads 4 bytes back)

    ``out`` (and everything in ``g.outputs``) is a static buffer that the next call overwrites.  ``width`` is 512 (the reference
    canvas) or any multiple of 64 above it up to pipeline.WIDE_MAX_WIDTH (wide lines: ``lq`` is the canvas restore_wide_image
    builds, locs are in units of ``width``, and ``outputs`` also holds ``seg``, the encoder segment of every character)."""

    def __init__(self, encoder, tspgan, sr, lines=1, chars=16, height=32, width=512, device=None, warmup=2, overlap_trunk=True):
        if device is None:
            device = next(encoder.parameters()).device
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("GraphedLines: the modules must live on a CUDA (sm_100a) device; there is no CPU fallback")
        if lines < 1 or chars < 1:
            raise RuntimeError("GraphedLines: lines and chars must be positive")
        from .pipeline import WIDE_ALIGN, WIDE_MAX_WIDTH, WIDE_SEGMENT
        if width < WIDE_SEGMENT or width % WIDE_ALIGN or width > WIDE_MAX_WIDTH:
            raise RuntimeError(f"GraphedLines: width {width} must be a multiple of {WIDE_ALIGN} in [{WIDE_SEGMENT}, {WIDE_MAX_WIDTH}]")
        self.encoder, self.tspgan, self.sr = encoder, tspgan, sr
        self.lines, self.chars, self.device, self.width = lines, chars, device, width
        self.segments = -(-width // WIDE_SEGMENT)
        if self.segments == 1:
            self._canvas = None
            self.lq = torch.zeros((lines, 3, height, width), dtype=torch.float32, device=device)
        else:
            # encoder input: the lines extended to whole 512-column segments with the canvas padding (-1 = the zero byte
            # normalised); lq is a view of its first ``width`` columns, so load() writes straight into it
            self._canvas = torch.full((lines, 3, height, self.segments * WIDE_SEGMENT), -1.0, dtype=torch.float32, device=device)
            self.lq = self._canvas[..., :width]
            self._line_first = torch.arange(0, (lines + 1) * chars, chars, dtype=torch.int32).to(device)
        self.labels = torch.zeros((lines * chars, 1), dtype=torch.int64, device=device)
        # default boxes: evenly spaced, so that warm-up and capture never see an empty window
        locs = torch.zeros((lines, 2 * chars), dtype=torch.float32)
        locs[:, 0::2] = (torch.arange(chars, dtype=torch.float32) + 0.5) / chars
        locs[:, 1::2] = 0.5 / chars
        self.locs = locs.to(device)
        self.flag = torch.zeros((1,), dtype=torch.int32, device=device)
        self.outputs = None
        # The SR decoder's LR trunk (networks.py:412-416) needs only the LR line: it is recorded on a second stream, as a parallel
        # branch of the graph, beside the encoder and the first (small-grid, latency-bound) generator layers.  Its convolutions
        # get their own split-K scratch so that the two branches never share one.
        self.overlap_trunk = bool(overlap_trunk)
        self._branch = torch.cuda.Stream(device=device) if self.overlap_trunk else None
        self._trunk_ws = torch.empty(ops._WS_BYTES // 4, dtype=torch.float32, device=device) if self.overlap_trunk else None
        self.graph = torch.cuda.CUDAGraph()
        self.launches = 0

        side = torch.cuda.Stream(device=device)
        side.wait_stream(torch.cuda.current_stream(device))
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(max(1, warmup)):        # packs weights, loads the tensor-map encoder, sizes the allocator
                self._step()
        torch.cuda.current_stream(device).wait_stream(side)
        torch.cuda.synchronize(device)
        l0 = ops.LAUNCHES
        # thread_local: other threads of the process (NCCL watchdog, NVML samplers) keep making CUDA calls during the capture
        with torch.cuda.graph(self.graph, capture_error_mode="thread_local"), torch.no_grad():
            self.outputs = self._step()
        self.launches = ops.LAUNCHES - l0

    def _step(self):
        with ops.deferred_checks(self.flag):
            self.flag.zero_()
            trunk, trunk_done, branch = None, None, None
            if self.overlap_trunk:
                branch = self._branch
                main = torch.cuda.current_stream(self.device)
                branch.wait_stream(main)
                with torch.cuda.stream(branch), ops.use_workspace(self._trunk_ws):
                    trunk = self.sr.trunk(self.lq)
                    trunk_done = torch.cuda.Event()
                    trunk_done.record(branch)
            # the encoder's classification / box branches and the generator's ToRGB chain also go to the second stream: the
            # generator only waits for w, the SR decoder only for the feature taps and the trunk
            enc_branch = (branch, self._trunk_ws) if branch is not None else None
            seg = None
            if self._canvas is None:      # the reference canvas: one segment, every character of line b gets w[b]
                logits, locs_lr, w = self.encoder(self.lq, _branch=enc_branch)
                styles = w.repeat_interleave(self.chars, dim=0)
            else:
                from .pipeline import WIDE_SEGMENT, _encoder_segments
                logits, locs_lr, w = self.encoder(_encoder_segments(self._canvas, self.segments), _branch=enc_branch)
                styles, seg = ops.char_segment_styles(w, self.locs, self._line_first, [self.chars] * self.lines, self.width,
                                                      self.segments, WIDE_SEGMENT)
            image, f64, f32_ = self.tspgan(styles=styles, labels=self.labels, noise=None, _branch=branch)
            n = self.chars
            p64 = [f64[b * n:(b + 1) * n] for b in range(self.lines)]
            p32 = [f32_[b * n:(b + 1) * n] for b in range(self.lines)]
            if trunk is not None:
                main.wait_event(trunk_done)
                trunk.record_stream(main)
            out = self.sr(self.lq, p64, p32, self.locs, _trunk=trunk)
            if branch is not None:
                main.wait_stream(branch)                       # joins logits / locs and the prior image
        outs = dict(sr=out, prior=image, fea64=f64, fea32=f32_, logits=logits, locs_lr=locs_lr, w=w)
        if seg is not None:
            outs["seg"] = seg
        return outs

    def load(self, lq=None, labels=None, locs=None):
        """Copy new inputs (host or device tensors) into the static buffers on the current stream."""
        if lq is not None:
            self.lq.copy_(lq, non_blocking=True)
        if labels is not None:
            self.labels.copy_(labels.reshape(self.labels.shape), non_blocking=True)
        if locs is not None:
            self.locs.copy_(locs, non_blocking=True)

    def replay(self):
        self.graph.replay()
        return self.outputs["sr"]

    def __call__(self, lq=None, labels=None, locs=None):
        self.load(lq, labels, locs)
        return self.replay()

    def check(self):
        """Synchronising read of the deferred error bits of the last replay; raises like the eager modules."""
        ops.raise_deferred(int(self.flag.item()))
        ops.check_range(self.device)        # fp16-range guard: the captured precision plan is baked in -- build a new GraphedLines after it fires

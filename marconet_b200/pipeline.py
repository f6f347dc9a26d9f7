"""Self-contained line-restoration flow on top of the three modules (SURVEY.md section 8f rows n3 / n4).

The reference's ``test_sr.py`` takes character labels and boxes from a third-party YOLO + OCR front-end; the original
single-model flow uses the encoder's own predictions instead: CTC-style de-duplicated argmax labels (test_w.py:34-40) and
boxes converted from the encoder's (left, right) pairs to (centre, half-width) exactly as the training model does
(Train/tspgan/models/tspgan_model.py:331-337).  Integer outputs (labels) are computed on the host, bit-exactly like the
reference; everything numeric runs through the module API (and therefore through the CUDA kernels).
"""
import collections

import torch

ALPHABET_SIZE = 6735          # classes [0, 6735) are characters, 6735 is the CTC blank (utils/alphabets.py, test_w.py:38)


def decode_labels(logits_row, n_alphabet=ALPHABET_SIZE):
    """argmax over classes, drop repeats and blanks (reference test_w.py:34-40).  ``logits_row``: [T, 6736]."""
    idx = torch.max(logits_row.detach(), 1)[1].cpu()
    out = []
    for i in range(idx.shape[0]):
        if not (i > 0 and idx[i - 1] == idx[i]) and idx[i] < n_alphabet:
            out.append(int(idx[i]))
    return out


def lr_to_center_halfwidth(locs_lr):
    """(left, right) pairs -> (centre, half-width) pairs, fp32, as Train/tspgan/models/tspgan_model.py:331-337."""
    out = locs_lr.clone()
    out[:, 0::2] = (locs_lr[:, 1::2] + locs_lr[:, 0::2]) / 2.0
    out[:, 1::2] = (locs_lr[:, 1::2] - locs_lr[:, 0::2]) / 2.0
    return out


def load_checkpoint(model, path_or_dict, prefer_ema=True, strict=True):
    """Load a reference-format checkpoint into one of the three modules.

    Accepts the released files' layout ``{'params': sd}`` (test_sr.py:43-51), BasicSR training checkpoints that also carry
    ``'params_ema'`` (Train/options/train.yml:69 uses it for the generator), a bare state_dict, and DDP ``module.`` prefixes."""
    ck = torch.load(path_or_dict, map_location="cpu") if isinstance(path_or_dict, (str, bytes)) or hasattr(path_or_dict, "read") else path_or_dict
    if isinstance(ck, dict) and ("params" in ck or "params_ema" in ck):
        key = "params_ema" if (prefer_ema and "params_ema" in ck) else ("params" if "params" in ck else "params_ema")
        ck = ck[key]
    sd = {(k[7:] if k.startswith("module.") else k): v for k, v in ck.items()}
    return model.load_state_dict(sd, strict=strict)


@torch.no_grad()
def restore_lines(encoder, tspgan, sr, lq, labels=None, locs=None, max_chars=16, check_range=True):
    """LQ lines [B,3,32,512] -> dict(sr, prior, labels, locs, w, logits).

    labels: optional list (per line) of int64 [n_b, 1] tensors; default = the encoder's decoded labels (at most ``max_chars``).
    locs:   optional [B, 2*n] (centre, half-width) in units of the line width; default = converted encoder boxes.
    check_range: synchronise at the end and look at the fp16-range flags (ops.poll_range); when a tensor-core conv overflowed the
    fp16 hi/lo split its layer is re-routed to the bf16 split and the step is re-run (at most 3 times) -- the caller never sees
    the Inf/NaN result."""
    if check_range:
        from . import ops
        for attempt in range(4):
            out = restore_lines(encoder, tspgan, sr, lq, labels, locs, max_chars, check_range=False)
            torch.cuda.synchronize(lq.device)
            if not ops.poll_range(lq.device) or attempt == 3:
                return out
    logits, locs_lr, w = encoder(lq)
    if labels is None:
        labels = []
        for b in range(lq.shape[0]):
            lab = decode_labels(logits[b])[:max_chars]
            labels.append(torch.tensor(lab, dtype=torch.long).reshape(-1, 1))
    if locs is None:
        locs = lr_to_center_halfwidth(locs_lr)
    counts = [int(l.shape[0]) for l in labels]
    total = sum(counts)
    p64, p32, priors = [], [], []
    if total > 0:
        styles = torch.cat([w[b:b + 1].expand(counts[b], -1) for b in range(lq.shape[0]) if counts[b] > 0], dim=0)
        lab_all = torch.cat([l for l in labels if l.shape[0] > 0], dim=0)
        img, f64, f32_ = tspgan(styles=styles, labels=lab_all, noise=None)       # one generator call for every character
        o = 0
        for n in counts:
            p64.append(f64[o:o + n]); p32.append(f32_[o:o + n]); priors.append(img[o:o + n]); o += n
    else:
        dev = lq.device
        for _ in counts:
            p64.append(torch.zeros(0, 256, 64, 64, device=dev)); p32.append(torch.zeros(0, 512, 32, 32, device=dev))
            priors.append(torch.zeros(0, 3, 128, 128, device=dev))
    out = sr(lq, p64, p32, locs)
    return dict(sr=out, prior=priors, labels=labels, locs=locs, w=w, logits=logits)


def boxes_to_locs(boxes, h, lq_width=512):
    """test_sr.py:118-134: detector boxes [x1, y1, x2, y2] in the ORIGINAL image -> locs [1, 2n] (centre, half-width) in units of
    the LQ canvas width.  Python-float arithmetic exactly as the script, stored as fp32."""
    locs = torch.zeros(1, len(boxes) * 2, dtype=torch.float32)
    for i, box in enumerate(boxes):
        x1, _, x2, _ = [float(v) for v in box]
        center, width = (x1 + x2) / 2.0, (x2 - x1) / 2.0
        locs[0, 2 * i] = (center * 32.0 / h) / lq_width
        locs[0, 2 * i + 1] = (width * 32.0 / h) / lq_width
    return locs


@torch.no_grad()
def restore_image(encoder, tspgan, sr, img_u8, labels, boxes):
    """One text-line image end to end on the device (the body of test_sr.py's loop, :98-201, with the labels / boxes the
    detector and OCR produced): uint8 [h, w, 3] image (host numpy / tensor or CUDA tensor) -> dict(sr_u8 [128, W, 3] uint8 bytes
    as cv2.imwrite would store them, cropped to the line's width; sr fp32; lq; lq_width).
    Pre- and post-processing run as CUDA kernels (mn_preprocess_lq_u8 / mn_postprocess_sr_u8)."""
    from . import ops
    dev = next(encoder.parameters()).device
    img = torch.as_tensor(img_u8)
    h = img.shape[0]
    img = img.to(dev, non_blocking=True).contiguous()
    lq, lq_w = ops.preprocess_lq(img)
    locs = boxes_to_locs(boxes, h, lq.shape[-1]).to(dev)
    _, _, w = encoder(lq)
    lab = torch.as_tensor(labels, dtype=torch.long).reshape(-1, 1)
    if lab.shape[0] == 0:
        raise ValueError("no character labels (test_sr.py:160-162 skips such images)")
    img_prior, f64, f32_ = tspgan(styles=w[:1].repeat(lab.shape[0], 1), labels=lab, noise=None)
    out = sr(lq, [f64], [f32_], locs)
    show_w = ops.round_half_even(img.shape[1] * (128 / h))    # ShowLQ = cv2.resize(img, fx=128/h, ...) (test_sr.py:98)
    sr_u8 = ops.postprocess_sr(out)[0, :, :show_w]            # ShowSR = sr[:, :ShowLQ.shape[1]] (test_sr.py:201)
    return dict(sr_u8=sr_u8, sr=out, lq=lq, lq_width=lq_w, prior=img_prior, locs=locs)


# ---------------------------------------------------------------------------------------------------------------------
# Lines wider than 512 LR columns (DESIGN.md "Wide lines").  The reference script pastes the 32-px-high line onto a 32x512 canvas
# and skips anything wider (test_sr.py:104-110).  Only the encoder is fixed at 512 columns (TextViT: 64 tokens); TSPSRNet is
# width-generic (its window integers use the map's own width, networks.py:426,435,460,469).  So the line is restored in ONE
# SR pass on a wider canvas, and the encoder runs on 512-column segments of it, each character taking the style of the
# segment that holds its centre.
# ---------------------------------------------------------------------------------------------------------------------
WIDE_SEGMENT = 512          # encoder input width (TextViT: 64 tokens of 8x8 patches over an 8x512 feature map)
WIDE_ALIGN = 64             # canvas width granularity: W/4 % 16 == 0 keeps every SR layer on the tcgen05 kernel (DESIGN 3.1)
# Largest canvas every kernel on the path can index: the biggest map is conv_final's up-sampled input, 128 channels at
# 128 x 4*Wsr pixels, and the elementwise / GroupNorm / conv epilogue kernels index maps with 32-bit element (or 4-element)
# counts (checked against 2^31 on the host, e.g. mn_resample_modulate, mn_groupnorm_apply, mn_conv2d_nhwc's M); 128*4*Wsr*128
# < 2^31 gives Wsr < 32768.  The owner tables (B*Wsr int32) and the preprocess canvas (3*32*S*512 floats) are far below it.
WIDE_MAX_WIDTH = ((2 ** 31 - 1) // (128 * 4 * 128)) // WIDE_ALIGN * WIDE_ALIGN          # 32704


# (Wr, Wsr, S, show_w) of one h x w image; compares equal to the plain tuple
WideGeometry = collections.namedtuple("WideGeometry", "lq_width canvas_width segments show_width")


def wide_geometry(h, w):
    """Canvas of an h x w line image, in Python floats as test_sr.py / cv::resize compute them:
      Wr     = round_half_even(w * (32/h))           the resized LQ width (cv2.resize with fx = 32/h, test_sr.py:99)
      Wsr    = max(512, 64 * ceil(Wr / 64))          the SR canvas, zero-padded on the right like the script's 512 canvas
      S      = ceil(Wsr / 512)                        encoder segments: canvas columns [512 s, 512 s + 512), zero-extended
      show_w = round_half_even(w * (128/h))          ShowLQ's width (test_sr.py:98); the output is sr[:, :show_w]
    Lines with Wr <= 512 get Wsr = 512, S = 1: exactly the script's canvas."""
    from .ops import round_half_even
    h, w = int(h), int(w)
    if h <= 0 or w <= 0:
        raise ValueError(f"empty image ({h} x {w})")
    wr = round_half_even(w * (32 / h))
    wsr = max(WIDE_SEGMENT, WIDE_ALIGN * (-(-wr // WIDE_ALIGN)))
    return WideGeometry(wr, wsr, -(-wsr // WIDE_SEGMENT), round_half_even(w * (128 / h)))


def _encoder_segments(canvas, segs):
    """[B, 3, 32, segs*512] canvas -> [B*segs, 3, 32, 512] (a strided view when B == 1; the encoder's NCHW->NHWC copy reads it)."""
    b, c, hh, _ = canvas.shape
    v = canvas.reshape(b, c, hh, segs, WIDE_SEGMENT).permute(0, 3, 1, 2, 4)
    return v[0] if b == 1 else v.reshape(b * segs, c, hh, WIDE_SEGMENT)


@torch.no_grad()
def wide_lines_forward(encoder, tspgan, sr, canvas, labels, locs, width, chars):
    """The wide-line data flow on preprocessed canvases: ``canvas`` fp32 [B, 3, 32, S*512] on the device (padding = -1, the
    normalised zero byte), ``labels`` int64 [B*chars, 1], ``locs`` fp32 device [B, 2*chars] in units of ``width`` (= Wsr, a
    multiple of 64, at least 512).  encoder on the B*S segments -> mn_char_segment_styles -> one TSPGAN call -> one TSPSRNet call
    on canvas[..., :width].  Returns dict(sr, prior, fea64, fea32, w, seg)."""
    from . import ops
    b = canvas.shape[0]
    segs = canvas.shape[-1] // WIDE_SEGMENT
    _, _, w = encoder(_encoder_segments(canvas, segs))
    first = torch.arange(0, (b + 1) * chars, chars, dtype=torch.int32).to(canvas.device, non_blocking=True)
    styles, seg = ops.char_segment_styles(w, locs, first, [chars] * b, width, segs, WIDE_SEGMENT)
    image, f64, f32_ = tspgan(styles=styles, labels=labels, noise=None)
    p64 = [f64[i * chars:(i + 1) * chars] for i in range(b)]
    p32 = [f32_[i * chars:(i + 1) * chars] for i in range(b)]
    out = sr(canvas[..., :width], p64, p32, locs)
    return dict(sr=out, prior=image, fea64=f64, fea32=f32_, w=w, seg=seg)


@torch.no_grad()
def restore_wide_image(encoder, tspgan, sr, img_u8, labels, boxes):
    """restore_image for a line of any width: uint8 [h, w, 3] image -> the same keys as restore_image plus ``segments`` (S),
    ``w`` ([S, 512], one style per encoder segment) and ``seg`` (int32 [n], the segment each character's style came from).

    The line is resized to height 32 (Wr columns) and pasted on a Wsr = max(512, 64*ceil(Wr/64)) canvas (wide_geometry); the
    encoder sees the S = ceil(Wsr/512) segments of it as one batch; character i takes w[seg_i] with seg_i the segment holding its
    32-level window centre; TSPGAN runs once for all characters and TSPSRNet once on [1, 3, 32, Wsr] -- no seams.  For Wr <= 512
    every step is restore_image's (same canvas, S = 1, every character gets w[0]), and the results are identical.
    Raises ValueError before launching anything when there are no labels or the canvas exceeds WIDE_MAX_WIDTH."""
    from . import ops
    img = torch.as_tensor(img_u8)
    if img.dim() != 3:
        raise ValueError(f"expected a uint8 [h, w, c] image, got shape {tuple(img.shape)}")
    h, w = int(img.shape[0]), int(img.shape[1])
    geo = wide_geometry(h, w)
    if geo.canvas_width > WIDE_MAX_WIDTH:
        raise ValueError(f"line of {h}x{w} px needs a {geo.canvas_width}-column LR canvas; at most {WIDE_MAX_WIDTH} columns fit the "
                         f"kernels' 32-bit indexing: crop it into shorter segments")
    lab = torch.as_tensor(labels, dtype=torch.long).reshape(-1, 1)
    n = lab.shape[0]
    if n == 0:
        raise ValueError("no character labels (test_sr.py:160-162 skips such images)")
    if len(boxes) < n:
        raise ValueError(f"{n} labels but only {len(boxes)} boxes")
    dev = next(encoder.parameters()).device
    img = img.to(dev, non_blocking=True).contiguous()
    canvas, lq_w = ops.preprocess_lq(img, out_w=geo.segments * WIDE_SEGMENT)
    locs = boxes_to_locs(boxes, h, geo.canvas_width).to(dev)
    out = wide_lines_forward(encoder, tspgan, sr, canvas, lab, locs, geo.canvas_width, n)
    sr_u8 = ops.postprocess_sr(out["sr"])[0, :, :geo.show_width]      # ShowSR = sr[:, :ShowLQ.shape[1]] (test_sr.py:201)
    return dict(sr_u8=sr_u8, sr=out["sr"], lq=canvas[..., :geo.canvas_width], lq_width=lq_w, prior=out["prior"], locs=locs,
                segments=geo.segments, w=out["w"], seg=out["seg"])


# ---------------------------------------------------------------------------------------------------------------------
# Per-layer precision plan (SURVEY.md section 8f row n4): fp16x3 / bf16x3 / fp32 and a power-of-two input scale per conv layer,
# chosen on calibration inputs against the exact fp32 kernels.  Needed the day real checkpoints replace the synthetic ones: the
# default fp16 hi/lo split (conv_tc2.cu) has fp32-grade mantissa but fp16's exponent range.
# ---------------------------------------------------------------------------------------------------------------------
def conv_layers(*modules):
    """Every ops.ConvWeight of the (already used, hence packed) modules, in pack order."""
    from . import ops
    out, seen = [], set()

    def walk(o):
        if isinstance(o, ops.ConvWeight):
            if id(o) not in seen:
                seen.add(id(o)); out.append(o)
        elif isinstance(o, dict):
            for v in o.values():
                walk(v)
        elif isinstance(o, (list, tuple)):
            for v in o:
                walk(v)

    for m in modules:
        for sub in m.modules():
            walk(getattr(sub, "_packed", None))
    return out


@torch.no_grad()
def tune_precision(encoder, tspgan, sr, lq, labels=None, locs=None, target_absmax=1024.0, fp32_fallback=1e-3, compare=True):
    """Calibrate the per-layer precision plan on (lq, labels, locs) -- representative LR lines -- and install it (ops.PLAN).

    pass 1 (range-safe bf16 split everywhere): max |input| of every tensor-core conv -> x_scale = 2^k with
            |x| * x_scale ~ ``target_absmax`` (64x headroom below 65504, inputs down to 2^-24 * target keep full hi/lo precision);
    pass 2 (``compare``): every such layer also runs through the exact fp32 kernel and through both split formats; the format with
            the smaller relative max-abs error wins, and a layer whose best error still exceeds ``fp32_fallback`` (relative to its
            output's max) runs on the fp32 CUDA-core kernel;
    pass 3: the plan is verified -- one more step, no range flag may rise.
    Returns a list of dict(name, absmax, x_scale, precision, err_f16x3, err_bf16x3), one per tensor-core conv layer."""
    import math
    from . import ops
    dev = lq.device
    with torch.cuda.device(dev):
        old_default = ops.default_precision()
        restore_lines(encoder, tspgan, sr, lq, labels, locs, check_range=False)     # packs the weights
        layers = conv_layers(encoder, tspgan, sr)
        for cw in layers:
            cw.set_plan(x_scale=1.0)
            cw.precision = None
            ops.PLAN[cw.name] = (None, 1.0)
        ops.PLAN_VERSION += 1
        try:
            ops.set_default_precision(ops.PREC_BF16X3_TC)
            with ops.calibration(dev) as cal:
                restore_lines(encoder, tspgan, sr, lq, labels, locs, check_range=False)
            res = cal.results()
        finally:
            ops.set_default_precision(old_default)
        ops.poll_range(dev, reroute=False)
        for cw, r in res.items():
            a = r["absmax"]
            k = 0 if not (a > 0 and math.isfinite(a)) else max(-24, min(24, round(math.log2(target_absmax / a))))
            cw.set_plan(x_scale=2.0 ** k)
        errs = {}
        if compare:
            with ops.calibration(dev, compare=True) as cal:
                restore_lines(encoder, tspgan, sr, lq, labels, locs, check_range=False)
            errs = cal.results()
            ops.poll_range(dev, reroute=False)
        report = []
        for cw, r in res.items():
            e = errs.get(cw, {})
            e16, ebf = e.get("err_f16x3", float("nan")), e.get("err_bf16x3", float("nan"))
            prec = ops.PREC_F16X3_TC
            if compare and cw in errs:
                prec = ops.PREC_F16X3_TC if (e16 <= ebf or not math.isfinite(ebf)) and math.isfinite(e16) else ops.PREC_BF16X3_TC
                if not (min(e16, ebf) <= fp32_fallback):
                    prec = ops.PREC_FP32_SIMT
            cw.set_plan(precision=prec)
            report.append(dict(name=cw.name, absmax=r["absmax"], x_scale=cw.x_scale, precision=prec, err_f16x3=e16, err_bf16x3=ebf))
        restore_lines(encoder, tspgan, sr, lq, labels, locs, check_range=False)
        torch.cuda.synchronize(dev)
        ops.check_range(dev)
    return report


def save_precision_plan(path):
    """ops.PLAN -> JSON {layer name: [precision or null, x_scale]}."""
    import json
    from . import ops
    with open(path, "w") as f:
        json.dump({k: [v[0], v[1]] for k, v in ops.PLAN.items()}, f, indent=1, sort_keys=True)


def load_precision_plan(path_or_dict, *modules):
    """Install a saved plan; already-packed layers of ``modules`` are updated in place, later packs pick it up by name."""
    import json
    from . import ops
    plan = json.load(open(path_or_dict)) if isinstance(path_or_dict, str) else path_or_dict
    for k, (prec, xs) in plan.items():
        ops.PLAN[k] = (None if prec is None else int(prec), float(xs))
    for cw in conv_layers(*modules):
        if cw.name in ops.PLAN:
            cw.precision, cw.x_scale = ops.PLAN[cw.name]
    ops.PLAN_VERSION += 1
    return plan

"""CPU restatement of the wide-line flow (TEST INFRASTRUCTURE ONLY): marconet_b200.pipeline.restore_wide_image on top of the
module restatements of oracle/restate.py (DESIGN.md "Wide lines").

The reference script pastes a line resized to height 32 onto a 32x512 canvas and skips wider lines (test_sr.py:104-110).  This
keeps every per-step rule of the script -- cv2 resize, zero-byte canvas, ToTensor + Normalize (oracle/image_ops.py), the box ->
locs arithmetic (:118-134), the ShowLQ crop (:98,201) -- and only widens the canvas: the SR module runs on Wsr columns (its
window integers use the map's own width, networks.py:426,435,460,469), the encoder on the 512-column segments, and every
character takes the style of the segment that holds its 32-level window centre.  No dependency on ``marconet_b200``.
"""
import math

import torch

from . import restate

SEGMENT = 512


def wide_geometry(h, w):
    """(Wr, Wsr, S, show_w): resized LQ width (cv::resize rounding of w*(32/h), test_sr.py:99), SR canvas width
    max(512, 64*ceil(Wr/64)), encoder segments ceil(Wsr/512), ShowLQ width (test_sr.py:98)."""
    wr = int(round(w * (32 / h)))                 # Python round(): half to even, as cvRound
    wsr = max(SEGMENT, 64 * math.ceil(wr / 64))
    return wr, wsr, math.ceil(wsr / SEGMENT), int(round(w * (128 / h)))


def char_segment(loc_center, width_total, segs):
    """Encoder segment of one character: the 32-level window centre (networks.py:426, fp32 multiply + truncation, as
    char_window) floor-divided by 512 and clamped into [0, segs)."""
    center = int((loc_center.float() * width_total).int())
    return min(max(center // SEGMENT, 0), segs - 1)


def boxes_to_locs(boxes, h, lq_width):
    """test_sr.py:118-134: detector boxes (original pixels) -> fp32 [1, 2n] (centre, half-width) in units of lq_width."""
    locs = torch.zeros(1, len(boxes) * 2, dtype=torch.float32)
    for i, (x1, _, x2, _) in enumerate(boxes):
        x1, x2 = float(x1), float(x2)
        locs[0, 2 * i] = ((x1 + x2) / 2.0 * 32.0 / h) / lq_width
        locs[0, 2 * i + 1] = ((x2 - x1) / 2.0 * 32.0 / h) / lq_width
    return locs


def wide_line(sds, img, labels, boxes, dtype=torch.float32):
    """One wide line image end to end: uint8 [h, w, 3] numpy image, labels (n ints), boxes (n x [x1, y1, x2, y2])."""
    from . import image_ops
    h, w = img.shape[:2]
    wr, wsr, segs, show_w = wide_geometry(h, w)
    canvas, lq_w = image_ops.preprocess_lq(img, out_w=segs * SEGMENT)      # zero-byte padding past Wr, as the script's canvas
    canvas = torch.from_numpy(canvas)
    seg_in = canvas[0].reshape(3, 32, segs, SEGMENT).permute(2, 0, 1, 3).contiguous()
    _, _, wst = restate.encoder_forward(sds["encoder"], seg_in, dtype)
    locs = boxes_to_locs(boxes, h, wsr)
    n = len(labels)
    seg = [char_segment(locs[0][2 * i], wsr, segs) for i in range(n)]
    lab = torch.tensor(list(labels), dtype=torch.long).reshape(-1, 1)
    prior, f64, f32_ = restate.tspgan_forward(sds["tspgan"], wst[seg], lab, dtype)
    lq = canvas[..., :wsr].contiguous()
    sr = restate.tspsr_forward(sds["sr"], lq, [f64], [f32_], locs, dtype)
    sr_u8 = image_ops.postprocess_sr(sr.float().numpy())[0, :, :show_w]
    windows = [restate.char_window(locs[0][2 * i], wsr, 16) + restate.char_window(locs[0][2 * i], 2 * wsr, 32) for i in range(n)]
    return dict(lq_width=wr, canvas_width=wsr, segments=segs, show_width=show_w, lq=lq, locs=locs, w=wst, seg=seg,
                prior=prior, fea64=f64, fea32=f32_, sr=sr, sr_u8=sr_u8, windows=windows, resized_width=lq_w)

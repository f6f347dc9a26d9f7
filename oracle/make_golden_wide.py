"""Generate tests/golden/wide_lines.npz from the UNMODIFIED reference modules (build container only).

    python -m oracle.make_golden_wide

Lines wider than the reference script's 512-column canvas (marconet_b200.pipeline.restore_wide_image): the reference modules
run on the wide canvas exactly as test_sr.py runs them on the 512 one -- the encoder on the 512-column segments as one batch,
TSPGAN once with each character's segment style, TSPSRNet once on [1, 3, 32, Wsr] -- with oracle/image_ops for the script's
cv2 / torchvision pre- and post-processing.  The geometry and segment rule come from oracle/restate_wide.py (restated there from
the pipeline's definition).  Stores the integers whole and strided samples of the float outputs (< 500 KB).
TEST INFRASTRUCTURE ONLY.
"""
import os

import numpy as np
import torch

from . import image_ops, ref_harness, restate, restate_wide, synth
from .make_golden import GOLDEN_DIR, golden_threads, sample

STRIDES = dict(prior=251, fea64=4099, fea32=2053, sr=257, sr_u8=97)


def wide_cases():
    """name -> dict(img uint8 [h, w, 3], labels [n], boxes [n][4], seed).  Shared with the tests."""
    out = {}
    # A: h = 32, w = 600 -> Wr 600, Wsr 640, S 2; 12 regular boxes, one of them across LQ column 512
    rng = np.random.default_rng(600)
    boxes = [[50 * i + 3, 2, 50 * i + 47, 30] for i in range(12)]
    out["A"] = dict(img=rng.integers(0, 256, (32, 600, 3), dtype=np.uint8), labels=synth.make_labels(12, 60).reshape(-1).tolist(),
                    boxes=boxes, seed=600)
    # B: h = 40, w = 1500 -> Wr 1200, Wsr 1216, S 3; 24 boxes: the first clipped at the left edge, one centred on LQ column
    # 512 (the segment border), one pair of overlapping windows, the last clipped at the canvas' right edge
    rng = np.random.default_rng(1500)
    boxes = [[0, 2, 20, 38]]
    for i in range(1, 22):
        boxes.append([62.5 * i + 6, 3, 62.5 * i + 56, 37])
    boxes[10] = [615, 3, 665, 37]                                   # centre 640 px -> LQ 512.0
    boxes.insert(16, [62.5 * 15 + 31, 4, 62.5 * 15 + 81, 36])       # 25 px (20 LQ columns) right of box 15: windows overlap
    boxes.append([1480, 2, 1540, 38])                               # centre beyond the image: LQ 1208, 32-level x2 clipped at 1216
    img = rng.integers(0, 256, (40, 1500, 3), dtype=np.uint8)
    img[:, ::7] //= 3                                                # some vertical structure
    out["B"] = dict(img=img, labels=synth.make_labels(24, 61).reshape(-1).tolist(), boxes=boxes, seed=1500)
    return out


def run_reference(models, case):
    """The reference modules on the wide canvas (test_sr.py:98-201 data flow with the canvas widened)."""
    img, labels, boxes = case["img"], case["labels"], case["boxes"]
    h, w = img.shape[:2]
    wr, wsr, segs, show_w = restate_wide.wide_geometry(h, w)
    canvas, lq_w = image_ops.preprocess_lq(img, out_w=segs * restate_wide.SEGMENT)
    assert lq_w == wr
    canvas = torch.from_numpy(canvas)
    locs = restate_wide.boxes_to_locs(boxes, h, wsr)
    n = len(labels)
    seg = [restate_wide.char_segment(locs[0][2 * i], wsr, segs) for i in range(n)]
    with torch.no_grad():
        _, _, wst = models["encoder"](canvas[0].reshape(3, 32, segs, restate_wide.SEGMENT).permute(2, 0, 1, 3).contiguous())
        lab = torch.tensor(labels, dtype=torch.long).reshape(-1, 1)
        prior, f64, f32_ = models["tspgan"](styles=wst[seg], labels=lab, noise=None)
        sr = models["sr"](canvas[..., :wsr].contiguous(), [f64], [f32_], locs)
    sr_u8 = image_ops.postprocess_sr(sr.numpy())[0, :, :show_w]
    windows = [restate.char_window(locs[0][2 * i], wsr, 16) + restate.char_window(locs[0][2 * i], 2 * wsr, 32) for i in range(n)]
    return dict(geometry=(wr, wsr, segs, show_w), w=wst, seg=seg, prior=prior, fea64=f64, fea32=f32_, sr=sr, sr_u8=sr_u8,
                windows=windows)


def record(name, case, out):
    """Fixture entries of one case (keys prefixed with the case name); also used by the tests to compare a fresh run."""
    g = out["geometry"]
    rec = dict(seed=np.int64(case["seed"]), boxes=np.asarray(case["boxes"], np.float64), labels=np.asarray(case["labels"], np.int64),
               geometry=np.asarray(g, np.int64), seg=np.asarray(out["seg"], np.int64), w=out["w"].numpy().astype(np.float32),
               windows=np.asarray(out["windows"], np.int64), sr_u8=np.ascontiguousarray(out["sr_u8"]).reshape(-1)[::STRIDES["sr_u8"]].copy())
    for k in ("prior", "fea64", "fea32", "sr"):
        rec[k] = sample(out[k], STRIDES[k])
        rec["sum_" + k] = np.float64(out[k].double().sum().item())
    return {f"{name}_{k}": v for k, v in rec.items()}


def main():
    sds = synth.make_checkpoints(0)
    models = ref_harness.build_reference_models(sds)
    data = {}
    with golden_threads():
        for name, case in wide_cases().items():
            out = run_reference(models, case)
            data.update(record(name, case, out))
            print(name, "geometry", out["geometry"], "seg", out["seg"])
    path = os.path.join(GOLDEN_DIR, "wide_lines.npz")
    np.savez_compressed(path, **data)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()

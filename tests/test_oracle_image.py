"""Pins oracle/image_ops.py (the restatement of the OpenCV resize + the script's normalisation / byte conversion,
test_sr.py:98-111,198-201) against the committed golden outputs of the real cv2 and, when cv2 is importable, against cv2
itself on fresh random images.  Bit-exact: this is byte/integer work."""
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "resize_cubic.npz")


def test_resize_matches_golden_cv2_outputs():
    from oracle import image_ops
    from oracle.make_golden_image import CASES, make_image
    g = np.load(GOLDEN)
    for h, w, seed in CASES:
        img = make_image(h, w, seed)
        got = image_ops.resize_cubic_u8(img, 32 / h, 32 / h)
        ref = g[f"out_{h}x{w}"]
        assert got.shape == ref.shape and np.array_equal(got, ref), (h, w, int((got != ref).sum()))


def test_resize_matches_live_cv2_without_ipp():
    cv2 = pytest.importorskip("cv2")
    from oracle import image_ops
    was = cv2.ipp.useIPP()
    cv2.ipp.setUseIPP(False)
    try:
        rng = np.random.default_rng(7)
        for trial in range(12):
            h, w = int(rng.integers(8, 100)), int(rng.integers(16, 700))
            img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8) if trial % 2 else (rng.integers(0, 2, (h, w, 3)) * 255).astype(np.uint8)
            ref = cv2.resize(img, (0, 0), fx=32 / h, fy=32 / h, interpolation=cv2.INTER_CUBIC)
            got = image_ops.resize_cubic_u8(img, 32 / h, 32 / h)
            assert got.shape == ref.shape and np.array_equal(got, ref), (h, w)
    finally:
        cv2.ipp.setUseIPP(was)


def test_preprocess_matches_the_script_arithmetic():
    """ToTensor + Normalize exactly as torchvision does them (test_sr.py:110-111)."""
    import torch
    from oracle import image_ops
    from oracle.make_golden_image import make_image
    img = make_image(48, 300, 0)
    lq, width = image_ops.preprocess_lq(img)
    resized = image_ops.resize_cubic_u8(img, 32 / 48, 32 / 48)
    assert width == resized.shape[1] == 200 and lq.shape == (1, 3, 32, 512)
    canvas = np.zeros((32, 512, 3), np.uint8)
    canvas[:, :width] = resized
    t = torch.from_numpy(canvas).permute(2, 0, 1).contiguous().to(torch.float32).div(255)      # ToTensor
    t = t.sub(0.5).div(0.5)                                                                    # Normalize(0.5, 0.5)
    assert np.array_equal(lq[0], t.numpy())
    assert (lq[0, :, :, width:] == -1.0).all()
    with pytest.raises(ValueError):
        image_ops.preprocess_lq(make_image(32, 600, 1))      # wider than 512 after resizing: the script skips such images


def test_postprocess_bytes():
    from oracle import image_ops
    rng = np.random.default_rng(3)
    sr = rng.uniform(-1.3, 1.3, (2, 3, 8, 16)).astype(np.float32)
    sr[0, 0, 0, :4] = [-1.0, 1.0, 0.0, 1.0 / 255 - 1.0]
    out = image_ops.postprocess_sr(sr)
    assert out.dtype == np.uint8 and out.shape == (2, 8, 16, 3)
    ref = np.clip((sr * np.float32(0.5) + np.float32(0.5)).transpose(0, 2, 3, 1)[..., ::-1], 0, 1) * np.float32(255.0)
    assert np.array_equal(out, np.rint(ref).astype(np.uint8))
    assert out[0, 0, 0, 2] == 0 and out[0, 0, 1, 2] == 255       # channel 0 lands in the last byte (flip)


def test_oracle_reproduces_the_reference_script_png_row(checkpoints):
    """uint8 image -> oracle pre-processing -> oracle nets -> oracle post-processing equals, byte for byte, the SR row of the PNG
    the UNMODIFIED reference test_sr.py wrote on the CPU (tests/golden/script_sr_row.npz, oracle/make_golden_script.py)."""
    import torch
    from marconet_b200 import pipeline
    from oracle import image_ops, restate
    from oracle.make_golden import golden_threads
    g = np.load(os.path.join(os.path.dirname(GOLDEN), "script_sr_row.npz"))
    img, boxes, labels, stride = g["image_rgb"], g["boxes"], g["labels"], int(g["stride"])
    lq, lq_w = image_ops.preprocess_lq(img)
    assert lq_w == 256
    lq_t = torch.from_numpy(lq)
    locs = pipeline.boxes_to_locs(boxes.tolist(), img.shape[0], 512)
    lab = torch.from_numpy(labels).reshape(-1, 1)
    with golden_threads():
        _, _, w = restate.encoder_forward(checkpoints["encoder"], lq_t)
        _, f64, f32_ = restate.tspgan_forward(checkpoints["tspgan"], w[:1].repeat(lab.shape[0], 1), lab)
        sr = restate.tspsr_forward(checkpoints["sr"], lq_t, [f64], [f32_], locs)
    row = image_ops.postprocess_sr(sr.numpy())[0, :, :1024]
    assert np.array_equal(row[::stride, ::stride], g["sr_row"])

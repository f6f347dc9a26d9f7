"""Lines wider than 512 LR columns on the B200 (pipeline.restore_wide_image, GraphedLines(width=...), mn_char_segment_styles)
against restore_image, the oracle restatement and the fixture made by the unmodified reference modules
(tests/golden/wide_lines.npz, oracle/make_golden_wide.py)."""
import os
import re

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "wide_lines.npz")
TOL = 1e-3


def _samp(t, stride):
    return t.detach().float().cpu().reshape(-1)[::stride].numpy()


def _models(gpu_models):
    return gpu_models["encoder"], gpu_models["tspgan"], gpu_models["sr"]


def _u8_close(got, ref):
    diff = np.abs(got.astype(int) - ref.astype(int))
    assert diff.max() <= 1 and (diff != 0).mean() < 0.15, (int(diff.max()), float((diff != 0).mean()))


def test_short_lines_reduce_to_restore_image(gpu_models):
    """Wr <= 512: the same canvas, S = 1, every character styled with w[0] -- byte and bit identical to restore_image."""
    from marconet_b200 import pipeline
    rng = np.random.default_rng(11)
    for h, w, n in ((40, 500, 4), (32, 512, 6), (24, 130, 2)):
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        labels = [int(v) for v in rng.integers(0, 6735, n)]
        boxes = [[w * i / n + 1, 2, w * (i + 1) / n - 1, h - 2] for i in range(n)]
        a = pipeline.restore_image(*_models(gpu_models), img, labels, boxes)
        b = pipeline.restore_wide_image(*_models(gpu_models), img, labels, boxes)
        assert b["segments"] == 1 and b["w"].shape == (1, 512) and b["seg"].tolist() == [0] * n
        for k in ("sr_u8", "sr", "lq", "prior", "locs"):
            assert a[k].shape == b[k].shape and torch.equal(a[k], b[k]), k
        assert a["lq_width"] == b["lq_width"]


@pytest.mark.parametrize("name", ["A", "B"])
def test_wide_line_vs_reference_golden(gpu_models, name):
    from marconet_b200 import pipeline
    from marconet_b200.models.networks import char_windows
    from oracle.make_golden_wide import STRIDES, wide_cases
    g = np.load(GOLDEN)
    case = wide_cases()[name]
    res = pipeline.restore_wide_image(*_models(gpu_models), case["img"], case["labels"], case["boxes"])
    wr, wsr, segs, show_w = g[f"{name}_geometry"].tolist()
    assert (res["lq_width"], res["lq"].shape[-1], res["segments"]) == (wr, wsr, segs)
    assert res["seg"].cpu().tolist() == g[f"{name}_seg"].tolist()
    n = len(case["labels"])
    w32, _, _ = char_windows(res["locs"].cpu(), [n], wsr, 16)
    w64, _, _ = char_windows(res["locs"].cpu(), [n], 2 * wsr, 32)
    # (line, x1, x2, y1) per level -> the fixture's (x1, x2, y1, y2) pairs
    got = [(a[1], a[2], a[3], a[3] + a[2] - a[1]) + (b[1], b[2], b[3], b[3] + b[2] - b[1]) for a, b in zip(w32, w64)]
    assert got == [tuple(r) for r in g[f"{name}_windows"].tolist()]
    errs = dict(w=float(np.abs(res["w"].cpu().numpy() - g[f"{name}_w"]).max()))
    for k in ("prior", "sr"):
        errs[k] = float(np.abs(_samp(res[k], STRIDES[k]) - g[f"{name}_{k}"]).max())
    print(name, "max-abs err vs reference golden:", errs)
    assert max(errs.values()) <= TOL, errs
    u8 = res["sr_u8"].cpu().numpy()
    assert u8.shape == (128, min(show_w, 4 * wsr), 3)
    _u8_close(np.ascontiguousarray(u8).reshape(-1)[::STRIDES["sr_u8"]], g[f"{name}_sr_u8"])


@pytest.mark.parametrize("name", ["A", "B"])
def test_wide_line_priors_vs_reference_golden(gpu_models, name):
    """The 64 / 32 px feature priors of the one generator call (styles from mn_char_segment_styles)."""
    from marconet_b200 import ops, pipeline
    from oracle.make_golden_wide import STRIDES, wide_cases
    g = np.load(GOLDEN)
    case = wide_cases()[name]
    enc, gen, sr = _models(gpu_models)
    h, w = case["img"].shape[:2]
    geo = pipeline.wide_geometry(h, w)
    dev = torch.device("cuda:0")
    canvas, _ = ops.preprocess_lq(torch.from_numpy(case["img"]).to(dev), out_w=geo.segments * 512)
    n = len(case["labels"])
    locs = pipeline.boxes_to_locs(case["boxes"], h, geo.canvas_width).to(dev)
    out = pipeline.wide_lines_forward(enc, gen, sr, canvas, torch.tensor(case["labels"]).reshape(-1, 1).to(dev), locs, geo.canvas_width, n)
    for k in ("fea64", "fea32"):
        err = float(np.abs(_samp(out[k], STRIDES[k]) - g[f"{name}_{k}"]).max())
        assert err <= TOL, (k, err)


@pytest.mark.parametrize("width", [256, 600, 1216, 2048])
def test_tspsrnet_other_widths_match_restatement(gpu_models, checkpoints, width):
    """The module at widths other than 512 against restate.tspsr_forward (width-generic like the reference module).  W = 600
    (W/4 not a multiple of 16) runs some layers on the fp32 kernel: only its correctness is checked here."""
    from oracle import restate, synth
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(width)
    lq = torch.randn(1, 3, 32, width, generator=g).clamp_(-1, 1)
    n = max(2, width // 64)
    styles = synth.make_styles(n, width)
    labels = synth.make_labels(n, width)
    _, f64, f32_ = restate.tspgan_forward(checkpoints["tspgan"], styles, labels)
    locs = torch.zeros(1, 2 * n)
    locs[0, 0::2] = (torch.arange(n, dtype=torch.float32) + 0.5) / n
    locs[0, 0] = 3.0 / width                        # clipped at the left edge
    locs[0, 2 * (n - 1)] = (width - 2.0) / width    # clipped at the right edge
    locs[0, 1::2] = 14.0 / width
    ref = restate.tspsr_forward(checkpoints["sr"], lq, [f64], [f32_], locs)
    got = gpu_models["sr"](lq.to(dev), [f64.to(dev)], [f32_.to(dev)], locs.to(dev))
    assert got.shape == ref.shape == (1, 3, 128, 4 * width)
    err = float((got.cpu() - ref).abs().max())
    print("width", width, "max-abs err", err)
    assert err <= TOL


def test_tspsrnet_rejects_what_the_reference_rejects_before_launching(gpu_models):
    from marconet_b200 import ops
    sr = gpu_models["sr"]
    dev = torch.device("cuda:0")
    p64, p32 = torch.zeros(1, 256, 64, 64, device=dev), torch.zeros(1, 512, 32, 32, device=dev)
    locs = torch.tensor([[0.5, 0.03]], device=dev)
    for shape, chars in (((1, 3, 32, 513), True), ((1, 3, 32, 514), True), ((1, 3, 32, 514), False), ((1, 3, 36, 512), True)):
        lq = torch.zeros(shape, device=dev)
        torch.cuda.synchronize()
        n0 = ops.LAUNCHES
        with pytest.raises(RuntimeError):
            if chars:
                sr(lq, [p64], [p32], locs)
            else:
                sr.trunk(lq)
        assert ops.LAUNCHES == n0, shape
    # H = 36 without characters is a valid reference call (no window is cut).  Its 36-, 18- and 9-row trunk layers are outside the
    # tensor-core geometry: they run on the exact fp32 kernel, logged with the planner's reason, and the line matches the fp32 path.
    lq36 = (torch.rand((1, 3, 36, 512), generator=torch.Generator().manual_seed(36)) * 2 - 1).to(dev)
    saved, prec = dict(ops.TC_FALLBACKS), ops.default_precision()
    try:
        ops.TC_FALLBACKS.clear()
        out = sr(lq36, [p64[:0]], [p32[:0]], locs[:, :0])
        h_rows = {v[0]: k[1] for k, v in ops.TC_FALLBACKS.items() if "H must be a multiple of 8" in v[2]}
        ops.set_default_precision(ops.PREC_FP32_SIMT)
        ref = sr(lq36, [p64[:0]], [p32[:0]], locs[:, :0])
    finally:
        ops.set_default_precision(prec)
        ops.TC_FALLBACKS.clear()
        ops.TC_FALLBACKS.update(saved)
    assert out.shape == ref.shape == (1, 3, 144, 2048)
    assert h_rows == {"sr.conv_body_32.0": 36, "sr.conv_body_32.2": 36, "sr.conv_body_16.0": 18, "sr.conv_body_16.2": 18,
                      "sr.conv_first_8.2": 9}, h_rows
    err = float((out - ref).abs().max())
    print("H = 36 line, tensor-core default vs fp32: max-abs", err)
    assert err <= TOL


def test_resample_modulate_checks_out_shape():
    from marconet_b200 import ops
    dev = torch.device("cuda:0")
    x = torch.zeros((1, 8, 129, 64), device=dev)
    bad = torch.zeros((1, 16, 257, 64), device=dev)            # one column short of the up-sampled 258
    n0 = ops.LAUNCHES
    with pytest.raises(RuntimeError, match="expected"):
        ops.resample_modulate(x, None, up=True, out=bad)
    assert ops.LAUNCHES == n0


def _restated_segments(locs, counts, width, segs):
    from oracle import restate_wide
    return [restate_wide.char_segment(locs[b][2 * c], width, segs) for b, n in enumerate(counts) for c in range(n)]


def test_char_segment_styles_kernel_adversarial_centres():
    from marconet_b200 import ops
    dev = torch.device("cuda:0")
    width, segs = 1216, 3
    w = torch.randn(2 * segs, 512, device=dev)
    centres = [[-0.3, -1e-7, 0.0, 511.0 / width, 512.0 / width, 1023.9 / width, 1024.0 / width, 1.0, 1.3],
               [0.5, 2.0, 1e-3, 600.0 / width, 0.0, 0.0, 0.0, 0.0, 0.0]]
    counts = [9, 4]
    locs = torch.zeros(2, 2 * 9)
    locs[:, 0::2] = torch.tensor(centres)
    first = torch.tensor([0, 9, 13], dtype=torch.int32, device=dev)
    want = _restated_segments(locs, counts, width, segs)
    rows = [b * segs + s for b, s in zip([0] * 9 + [1] * 4, want)]
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    for deferred in (False, True):
        with ops.deferred_checks(flag if deferred else None):
            styles, seg = ops.char_segment_styles(w, locs.to(dev), first, counts, width, segs)
        assert seg.cpu().tolist() == want
        assert torch.equal(styles, w[rows])
    assert int(flag.item()) == 0
    # one segment: every character gets its line's row (test_sr.py's w0.repeat(n, 1))
    styles, seg = ops.char_segment_styles(w[:2], locs.to(dev), first, counts, 512, 1)
    assert seg.cpu().tolist() == [0] * 13 and torch.equal(styles, w[:2][[0] * 9 + [1] * 4])


def test_wide_canvases_stay_on_the_tensor_cores(gpu_models):
    """At Wsr in {640, 1216, 2048} no conv shape falls back to the fp32 kernel for a layer the 512 path keeps on tcgen05.  The
    512 baseline includes the encoder on a 4-line batch: the wide flow's S segments are the same encoder batch as S lines of the
    512 path (its classification head, Cout = 6736, leaves the small-M linear above 64 rows).  Module graphs are off here: a
    replayed graph issues no conv2d call, so it would log nothing."""
    from marconet_b200 import ops, pipeline
    rng = np.random.default_rng(5)

    def layers_on_fallback(w_px):
        ops.TC_FALLBACKS.clear()
        img = rng.integers(0, 256, (32, w_px, 3), dtype=np.uint8)
        n = max(2, w_px // 32)
        boxes = [[w_px * i / n + 1, 2, w_px * (i + 1) / n - 1, 30] for i in range(n)]
        pipeline.restore_wide_image(*_models(gpu_models), img, [int(v) for v in rng.integers(0, 6735, n)], boxes)
        return {re.sub(r"#\d+", "", v[0]) for v in ops.TC_FALLBACKS.values()}     # unnamed weights carry a per-instance tag

    saved, graphs = dict(ops.TC_FALLBACKS), ops.MODULE_GRAPHS
    ops.MODULE_GRAPHS = False
    try:
        base = layers_on_fallback(500)
        ops.TC_FALLBACKS.clear()
        gpu_models["encoder"](torch.zeros((4, 3, 32, 512), device="cuda:0"))
        base |= {re.sub(r"#\d+", "", v[0]) for v in ops.TC_FALLBACKS.values()}
        for w_px in (600, 1200, 2048):
            extra = layers_on_fallback(w_px) - base
            assert not extra, (w_px, extra)
    finally:
        ops.MODULE_GRAPHS = graphs
        ops.TC_FALLBACKS.clear()
        ops.TC_FALLBACKS.update(saved)


def test_graphed_wide_lines_equal_eager_and_golden(gpu_models):
    """GraphedLines(width=1216, lines=2, chars=24): replays bit-identical to the eager wide-line data flow on the same inputs, and
    line 0 (golden case B) within 1e-3 of the reference fixture."""
    from marconet_b200 import ops, pipeline
    from marconet_b200.graph import GraphedLines
    from oracle.make_golden_wide import STRIDES, wide_cases
    g = np.load(GOLDEN)
    dev = torch.device("cuda:0")
    case = wide_cases()["B"]
    h, w = case["img"].shape[:2]
    geo = pipeline.wide_geometry(h, w)
    assert geo.canvas_width == 1216
    img1 = np.ascontiguousarray(case["img"][:, ::-1])                                  # second line: the mirrored image
    canv = [ops.preprocess_lq(torch.from_numpy(im).to(dev), out_w=geo.segments * 512)[0] for im in (case["img"], img1)]
    canvas = torch.cat(canv, 0)
    locs = torch.cat([pipeline.boxes_to_locs(case["boxes"], h, 1216),
                      pipeline.boxes_to_locs([[w - b[2], b[1], w - b[0], b[3]] for b in case["boxes"]], h, 1216)], 0).to(dev)
    labels = torch.tensor(case["labels"] + case["labels"][::-1]).reshape(-1, 1).to(dev)
    gl = GraphedLines(*_models(gpu_models), lines=2, chars=24, width=1216, device=dev)
    for _ in range(3):
        sr = gl(canvas[..., :1216], labels, locs)
        gl.check()
    got = {k: v.clone() for k, v in gl.outputs.items()}
    eager = pipeline.wide_lines_forward(*_models(gpu_models), canvas, labels, locs, 1216, 24)
    for k, v in eager.items():
        assert torch.equal(got[k], v), f"graph replay output '{k}' differs from the eager wide-line path"
    err = float(np.abs(_samp(sr[:1], STRIDES["sr"]) - g["B_sr"]).max())
    print("graphed wide line: sr max-abs err vs golden", err)
    assert err <= TOL
    assert got["seg"][:24].cpu().tolist() == g["B_seg"].tolist()


def test_graphed_lines_reject_unsupported_widths(gpu_models):
    from marconet_b200.graph import GraphedLines
    for width in (256, 513, 600, 32768):
        with pytest.raises(RuntimeError):
            GraphedLines(*_models(gpu_models), lines=1, chars=4, width=width)


def test_width_limit_raises_without_launching(gpu_models):
    from marconet_b200 import ops, pipeline
    n0 = ops.LAUNCHES
    img = np.zeros((64, 2 * (pipeline.WIDE_MAX_WIDTH + 64), 3), np.uint8)      # Wr = WIDE_MAX_WIDTH + 64
    with pytest.raises(ValueError):
        pipeline.restore_wide_image(*_models(gpu_models), img, [3], [[0, 0, 40, 64]])
    assert ops.LAUNCHES == n0

"""Wide lines on the host: canvas geometry, the segment rule, the width limit, and the oracle restatement against the fixture
made by the unmodified reference modules (tests/golden/wide_lines.npz, oracle/make_golden_wide.py)."""
import os

import numpy as np
import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "wide_lines.npz")


@pytest.mark.parametrize("h,w,expect", [((32), 600, (600, 640, 2, 2400)), (40, 1500, (1200, 1216, 3, 4800)),
                                        (40, 500, (400, 512, 1, 1600)), (80, 2561, (1024, 1024, 2, 4098))])
def test_wide_geometry(h, w, expect):
    from marconet_b200 import pipeline
    from oracle import restate_wide as restate
    g = pipeline.wide_geometry(h, w)
    assert g == expect and restate.wide_geometry(h, w) == expect
    assert (g.lq_width, g.canvas_width, g.segments, g.show_width) == expect
    # the output is sr_u8[:, :show_w] of a 4*Wsr-wide SR line: (80, 2561) keeps 4096 of its 4098 columns
    assert min(g.show_width, 4 * g.canvas_width) == len(range(4 * g.canvas_width)[:g.show_width])


def test_wide_geometry_short_lines_take_the_reference_canvas():
    from marconet_b200 import pipeline
    for h, w in ((32, 512), (32, 1), (17, 272), (100, 1600), (64, 1024)):
        g = pipeline.wide_geometry(h, w)
        assert g.lq_width <= 512 and g.canvas_width == 512 and g.segments == 1
    g = pipeline.wide_geometry(32, 513)
    assert g.canvas_width == 576 and g.segments == 2


def test_segment_rule_on_adversarial_centres():
    """Negative centres, exactly 512, at and beyond Wsr: clamp(floor(cen / 512), 0, S-1) with the fp32 product truncated."""
    from oracle import restate_wide as restate
    wsr, segs = 1216, 3
    cases = {-0.2: 0, -1e-9: 0, 0.0: 0, 511.0 / wsr: 0, 512.0 / wsr: None, 1023.9 / wsr: 1, 1024.0 / wsr: None, 1.0: 2, 1.7: 2}
    for loc, want in cases.items():
        t = torch.tensor(loc, dtype=torch.float32)
        cen = int((t * wsr).int())
        got = restate.char_segment(t, wsr, segs)
        assert got == min(max(cen // 512, 0), segs - 1)
        if want is not None:
            assert got == want, (loc, got)
    # a centre whose fp32 product lands exactly on 512 goes to segment 1, one just below to segment 0
    t = torch.tensor(0.5, dtype=torch.float32)
    assert restate.char_segment(t, 1024, 2) == 1
    assert restate.char_segment(torch.nextafter(t, torch.tensor(0.0)), 1024, 2) == 0


def test_width_limit_rejects_before_touching_the_modules():
    from marconet_b200 import pipeline
    assert pipeline.WIDE_MAX_WIDTH == 32704 and pipeline.WIDE_MAX_WIDTH % 64 == 0
    assert 128 * 4 * pipeline.WIDE_MAX_WIDTH * 128 < 2 ** 31 <= 128 * 4 * (pipeline.WIDE_MAX_WIDTH + 64) * 128

    class NoModule:
        def parameters(self):
            raise AssertionError("restore_wide_image touched the module before the width check")

    img = np.zeros((32, pipeline.WIDE_MAX_WIDTH + 1, 3), np.uint8)          # Wsr = WIDE_MAX_WIDTH + 64
    with pytest.raises(ValueError, match="crop"):
        pipeline.restore_wide_image(NoModule(), NoModule(), NoModule(), img, [1], [[0, 0, 10, 32]])


def _golden():
    return np.load(GOLDEN)


@pytest.mark.parametrize("name", ["A", "B"])
def test_restated_wide_line_reproduces_the_reference_fixture(name, checkpoints):
    from oracle import restate_wide as restate
    from oracle.make_golden import golden_threads
    from oracle.make_golden_wide import record, wide_cases
    g = _golden()
    case = wide_cases()[name]
    assert int(g[f"{name}_seed"]) == case["seed"]
    assert np.array_equal(g[f"{name}_labels"], np.asarray(case["labels"])) and np.array_equal(g[f"{name}_boxes"], np.asarray(case["boxes"]))
    with golden_threads():
        out = restate.wide_line(checkpoints, case["img"], case["labels"], case["boxes"])
    out["geometry"] = (out["lq_width"], out["canvas_width"], out["segments"], out["show_width"])
    rec = record(name, case, out)
    for k, v in rec.items():
        assert np.array_equal(v, g[k]), k
    expect = dict(A=(600, 640, 2, 2400), B=(1200, 1216, 3, 4800))[name]
    assert out["geometry"] == expect and out["resized_width"] == expect[0]
    assert out["sr_u8"].shape == (128, min(expect[3], 4 * expect[1]), 3)
    assert len(set(out["seg"])) == expect[2]           # every segment styles at least one character


@pytest.mark.skipif(not __import__("oracle.ref_harness", fromlist=["available"]).available(), reason="reference tree not present")
def test_restatement_bit_identical_to_reference_modules_at_width_600(checkpoints):
    """TSPSRNet of the unmodified reference at W = 600 (not a multiple of 64: its trunk takes any W = 0 mod 4) against
    restate.tspsr_forward, and the encoder on a two-segment batch against restate.encoder_forward."""
    from oracle import ref_harness, restate, synth
    from oracle.make_golden import golden_threads
    with golden_threads():
        ref = ref_harness.build_reference_models(checkpoints)
        g = torch.Generator().manual_seed(600)
        lq = torch.randn(1, 3, 32, 600, generator=g).clamp_(-1, 1)
        segs = torch.cat([lq[..., :512], torch.cat([lq[..., 512:], torch.full((1, 3, 32, 424), -1.0)], -1)], 0)
        with torch.no_grad():
            _, _, w_ref = ref["encoder"](segs)
        _, _, w_res = restate.encoder_forward(checkpoints["encoder"], segs)
        assert torch.equal(w_ref, w_res)
        labels = synth.make_labels(3, 7)
        locs = torch.tensor([[10.0 / 600, 0.02, 300.0 / 600, 0.02, 597.0 / 600, 0.02]])
        with torch.no_grad():
            _, f64, f32_ = ref["tspgan"](styles=w_ref[[0, 0, 1]], labels=labels, noise=None)
            sr_ref = ref["sr"](lq, [f64], [f32_], locs)
        sr_res = restate.tspsr_forward(checkpoints["sr"], lq, [f64], [f32_], locs)
    assert sr_ref.shape == (1, 3, 128, 2400)
    assert torch.equal(sr_ref, sr_res)

"""Module-level parity of the CUDA path (through the reference-facing module API) against the CPU oracle
and the committed golden fixtures (generated from the unmodified reference modules).

Tolerance: north_star states <= 1e-3 max-abs error on pixels/features, bit-exact integer outputs
(argmax labels, window integers).  The fp32 CUDA-core path is held to a much tighter bound.
"""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True, params=["fp16x3_tcgen05", "fp32_simt"])
def precision_mode(request):
    """Every module-level parity test runs on both conv paths: the default tcgen05 operand-split path and the
    exact fp32 CUDA-core path."""
    from marconet_b200 import ops
    old = ops.default_precision()
    ops.set_default_precision(ops.PREC_F16X3_TC if request.param == "fp16x3_tcgen05" else ops.PREC_FP32_SIMT)
    yield request.param
    ops.set_default_precision(old)

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TOL = 1e-3          # north_star budget (golden-fixture tests assert this)


def _tol_internal():
    """Tighter bound the module-vs-oracle tests hold each path to: 2e-4 for the fp32 CUDA-core path, 5e-4 for the
    tcgen05 operand-split path (its fp32 TMEM accumulation truncates; see conv_tc2.cu)."""
    from marconet_b200 import ops
    return 2e-4 if ops.default_precision() == ops.PREC_FP32_SIMT else 5e-4


def _maxerr(a, b):
    return (a.detach().float().cpu() - b.detach().float().cpu()).abs().max().item()


def test_tspgan_matches_oracle(gpu_models, checkpoints):
    from oracle import restate, synth
    dev = torch.device("cuda:0")
    n = 5
    labels, styles = synth.make_labels(n, 3), synth.make_styles(n, 3)      # distinct w per char: true per-sample modulation
    with torch.no_grad():
        img, f64, f32_ = gpu_models["tspgan"](styles=styles.to(dev), labels=labels, noise=None)   # labels stay on CPU like test_sr.py:180
    oi, o64, o32 = restate.tspgan_forward(checkpoints["tspgan"], styles, labels)
    assert img.shape == oi.shape and f64.shape == o64.shape and f32_.shape == o32.shape
    errs = (_maxerr(img, oi), _maxerr(f64, o64), _maxerr(f32_, o32))
    print("tspgan max-abs err (image, fea64, fea32):", errs)
    assert max(errs) <= _tol_internal()


def test_tspgan_two_labels_per_row_and_errors(gpu_models, checkpoints):
    from oracle import restate, synth
    dev = torch.device("cuda:0")
    labels = torch.tensor([[5, 6000], [17, 17]])
    styles = synth.make_styles(2, 5)
    img, f64, f32_ = gpu_models["tspgan"](styles.to(dev), labels.to(dev), None)
    oi, o64, o32 = restate.tspgan_forward(checkpoints["tspgan"], styles, labels)
    assert tuple(img.shape) == (2, 3, 128, 256)
    assert max(_maxerr(img, oi), _maxerr(f64, o64), _maxerr(f32_, o32)) <= _tol_internal()
    with pytest.raises(IndexError):           # unknown char -> alphabet.find == -1 (test_sr.py:24-29)
        gpu_models["tspgan"](styles.to(dev), torch.tensor([[-1, 3], [1, 2]]), None)
    with pytest.raises(IndexError):
        gpu_models["tspgan"](styles.to(dev), torch.tensor([[6736, 3], [1, 2]]), None)
    with pytest.raises(RuntimeError):         # CPU input: no fallback
        gpu_models["tspgan"](styles, labels, None)


def test_encoder_matches_oracle_and_argmax_exact(gpu_models, checkpoints):
    from oracle import restate, synth
    dev = torch.device("cuda:0")
    lq = synth.make_lq(2, 0)
    logits, locs, w = gpu_models["encoder"](lq.to(dev))
    ol, olo, ow = restate.encoder_forward(checkpoints["encoder"], lq)
    errs = (_maxerr(logits, ol), _maxerr(locs, olo), _maxerr(w, ow))
    print("encoder max-abs err (logits, locs, w):", errs)
    assert max(errs) <= _tol_internal()
    assert torch.equal(logits.argmax(-1).cpu(), ol.argmax(-1)), "char-index integers must be bit-exact"
    for b in range(2):
        assert restate.clear_labels(logits[b].cpu()) == restate.clear_labels(ol[b])


def test_sr_ragged_matches_oracle(gpu_models, checkpoints):
    """Clipped, overlapping, multi-line windows (the hard semantics of networks.py:425-448)."""
    from oracle import restate
    from oracle.make_golden import case_inputs
    dev = torch.device("cuda:0")
    inp = case_inputs("ragged")
    g = torch.Generator().manual_seed(77)
    p64 = [torch.randn(l.shape[0], 256, 64, 64, generator=g) for l in inp["labels"]]
    p32 = [torch.randn(l.shape[0], 512, 32, 32, generator=g) for l in inp["labels"]]
    sr = gpu_models["sr"](inp["lq"].to(dev), [p.to(dev) for p in p64], [p.to(dev) for p in p32], inp["locs"].to(dev))
    ref = restate.tspsr_forward(checkpoints["sr"], inp["lq"], p64, p32, inp["locs"])
    assert tuple(sr.shape) == (2, 3, 128, 2048)
    err = _maxerr(sr, ref)
    print("sr (ragged) max-abs err:", err)
    assert err <= _tol_internal()


def test_window_integers_bit_exact():
    from marconet_b200.models.networks import char_windows
    g = np.load(os.path.join(GOLDEN, "ragged.npz"))
    from oracle.make_golden import case_inputs
    inp = case_inputs("ragged")
    counts = [l.shape[0] for l in inp["labels"]]
    w32, _, _ = char_windows(inp["locs"], counts, 512, 16)
    w64, _, _ = char_windows(inp["locs"], counts, 1024, 32)
    got = [[a[1], a[2], a[3], a[3] + a[2] - a[1], b[1], b[2], b[3], b[3] + b[2] - b[1]] for a, b in zip(w32, w64)]
    assert np.array_equal(np.asarray(got, dtype=np.int64), g["windows"])


@pytest.mark.parametrize("name", ["config2", "ragged"])
def test_full_pipeline_vs_golden(gpu_models, name):
    """encoder -> TSPGAN -> TSPSRNet exactly as test_sr.py:145-197 drives them, against samples of the
    UNMODIFIED reference's outputs (tests/golden, made by oracle/make_golden.py)."""
    from oracle.make_golden import STRIDES, case_inputs
    dev = torch.device("cuda:0")
    g = np.load(os.path.join(GOLDEN, f"{name}.npz"))
    inp = case_inputs(name)
    lq = inp["lq"].to(dev)
    logits, enc_locs, w = gpu_models["encoder"](lq)
    imgs, p64, p32 = [], [], []
    for b in range(lq.shape[0]):
        lab = inp["labels"][b]
        img, f64, f32_ = gpu_models["tspgan"](styles=w[b:b + 1].repeat(lab.shape[0], 1), labels=lab, noise=None)
        imgs.append(img); p64.append(f64); p32.append(f32_)
    sr = gpu_models["sr"](lq, p64, p32, inp["locs"].to(dev))

    def samp(t, key):
        return t.detach().float().cpu().contiguous().reshape(-1)[::STRIDES[key]].numpy()

    got = dict(logits=samp(logits, "logits"), locs=samp(enc_locs, "locs"), w=samp(w, "w"),
               image=samp(torch.cat(imgs), "image"), fea64=samp(torch.cat(p64), "fea64"), fea32=samp(torch.cat(p32), "fea32"),
               sr=samp(sr, "sr"))
    errs = {k: float(np.abs(v - g[k]).max()) for k, v in got.items()}
    print(name, "max-abs err vs reference golden:", errs)
    assert max(errs.values()) <= TOL, errs
    assert np.array_equal(logits.argmax(-1).cpu().numpy(), g["argmax"])
    assert abs(float(sr.double().sum().item()) - float(g["sum_sr"])) <= 1e-3 * sr.numel() ** 0.5 + 1.0


def test_no_priors_and_shapes(gpu_models):
    """A line without characters: the SR trunk alone (priors lists empty for that line)."""
    from oracle import synth
    dev = torch.device("cuda:0")
    lq = synth.make_lq(1, 3).to(dev)
    sr = gpu_models["sr"](lq, [torch.zeros(0, 256, 64, 64, device=dev)], [torch.zeros(0, 512, 32, 32, device=dev)],
                          torch.zeros(1, 0, device=dev))
    assert tuple(sr.shape) == (1, 3, 128, 2048) and torch.isfinite(sr).all()


def test_style_interpolation_flow_like_test_w(gpu_models, checkpoints):
    """The reference's test_w.py:95-108 data flow: two encoder passes, labels = CTC-deduplicated argmax of image 1,
    priors generated for w = w1*t + w2*(1-t)."""
    from oracle import restate, synth
    dev = torch.device("cuda:0")
    lq1, lq2 = synth.make_lq(1, 21), synth.make_lq(1, 22)
    logits1, _, w1 = gpu_models["encoder"](lq1.to(dev))
    _, _, w2 = gpu_models["encoder"](lq2.to(dev))
    ol1, _, ow1 = restate.encoder_forward(checkpoints["encoder"], lq1)
    _, _, ow2 = restate.encoder_forward(checkpoints["encoder"], lq2)
    labels = restate.clear_labels(logits1[0].cpu())
    assert labels == restate.clear_labels(ol1[0]), "argmax / dedup labels must be bit-exact"
    labels = torch.tensor(labels[:4], dtype=torch.long).unsqueeze(1)      # first 4 characters keep the CPU oracle quick
    for t in (0.0, 0.3, 1.0):
        new_w = w1 * t + w2 * (1 - t)
        img, _, _ = gpu_models["tspgan"](styles=new_w.repeat(labels.size(0), 1), labels=labels, noise=None)
        oimg, _, _ = restate.tspgan_forward(checkpoints["tspgan"], (ow1 * t + ow2 * (1 - t)).repeat(labels.size(0), 1), labels)
        assert _maxerr(img, oimg) <= _tol_internal() * 2

"""CPU tests: the oracle restatement against the golden fixtures made from the UNMODIFIED reference
modules (tests/golden, oracle/make_golden.py)."""
import os

import numpy as np
import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_checkpoint_keys_and_digests(checkpoints):
    from oracle.make_golden import sd_digest
    assert (len(checkpoints["tspgan"]), len(checkpoints["encoder"]), len(checkpoints["sr"])) == (96, 124, 144)
    want = dict(l.split() for l in open(os.path.join(GOLDEN, "checkpoint_sha256.txt")))
    got = {k: sd_digest(v) for k, v in checkpoints.items()}
    # randn-derived tensors are bit-reproducible; the spectral-norm u/v come out of 30 mat-vec iterations whose
    # last bits may depend on the BLAS thread count, so only the non-SR digests are asserted exactly.
    assert got["tspgan"] == want["tspgan"] and got["encoder"] == want["encoder"]


def test_oracle_matches_reference_golden_ragged(checkpoints):
    """Small case (5 chars, 2 lines): restate.py vs samples of the reference modules' outputs."""
    from oracle import restate
    from oracle.make_golden import STRIDES, case_inputs, golden_threads
    g = np.load(os.path.join(GOLDEN, "ragged.npz"))
    inp = case_inputs("ragged")
    with golden_threads():
        out = restate.full_line(checkpoints, inp["lq"], inp["labels"], inp["locs"])
    samp = lambda t, k: t.reshape(-1)[::STRIDES[k]].numpy()
    errs = dict(
        logits=np.abs(samp(out["logits"], "logits") - g["logits"]).max(), w=np.abs(samp(out["w"], "w") - g["w"]).max(),
        locs=np.abs(samp(out["enc_locs"], "locs") - g["locs"]).max(),
        image=np.abs(samp(torch.cat(out["prior"]), "image") - g["image"]).max(),
        fea64=np.abs(samp(torch.cat(out["fea64"]), "fea64") - g["fea64"]).max(),
        fea32=np.abs(samp(torch.cat(out["fea32"]), "fea32") - g["fea32"]).max(),
        sr=np.abs(samp(out["sr"], "sr") - g["sr"]).max())
    assert max(errs.values()) <= 2e-5, errs        # same ops, same order: rounding noise only
    assert np.array_equal(out["logits"].argmax(-1).numpy(), g["argmax"])


def test_window_integers_golden():
    from oracle import restate
    from oracle.make_golden import case_inputs
    for name in ("config2", "ragged"):
        g = np.load(os.path.join(GOLDEN, f"{name}.npz"))
        inp = case_inputs(name)
        wins = []
        for b in range(inp["lq"].shape[0]):
            for c in range(inp["labels"][b].shape[0]):
                wins.append(restate.char_window(inp["locs"][b][2 * c], 512, 16) + restate.char_window(inp["locs"][b][2 * c], 1024, 32))
        assert np.array_equal(np.asarray(wins), g["windows"])
    # config 2: every window is full width
    assert (g["windows"][:, 1] - g["windows"][:, 0]).tolist() == [32] * 16 if name == "config2" else True


def test_clear_labels_ctc_dedup():
    from oracle import restate
    logits = torch.full((6, 6736), -1.0)
    for t, c in enumerate([5, 5, 6735, 5, 9, 9]):
        logits[t, c] = 1.0
    assert restate.clear_labels(logits) == [5, 5, 9]


def test_oracle_is_bit_identical_to_reference_modules(checkpoints):
    """restate.py vs the outputs of the unmodified reference modules (tests/golden/modules.npz, oracle/make_golden.py), with
    the thread count they were generated with.  TSPGAN takes the reference's stored w; TSPSRNet takes restate's own priors,
    which equal the reference's within the same bound."""
    from oracle import restate
    from oracle.make_golden import MODULE_STRIDES, golden_threads, modules_case, sample
    g = np.load(os.path.join(GOLDEN, "modules.npz"))
    with golden_threads(), torch.no_grad():
        lq, labels, locs = modules_case()
        ol, olo, ow = restate.encoder_forward(checkpoints["encoder"], lq)
        oi, o64, o32 = restate.tspgan_forward(checkpoints["tspgan"], torch.from_numpy(g["w"]).reshape(1, -1).repeat(2, 1), labels)
        os_ = restate.tspsr_forward(checkpoints["sr"], lq, [o64], [o32], locs)
    out = dict(logits=ol, locs=olo, w=ow, image=oi, fea64=o64, fea32=o32, sr=os_)
    for k, t in out.items():
        assert np.abs(sample(t, MODULE_STRIDES[k]) - g[k]).max() <= 1e-6, k

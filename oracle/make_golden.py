"""Generate tests/golden/*.npz from the UNMODIFIED reference modules (build container only).

    python -m oracle.make_golden

Runs /root/reference/models (via oracle/ref_harness.py) on the seeded synthetic
checkpoints and inputs of oracle/synth.py and stores strided samples of every
stage output plus the integer outputs (argmax labels, window integers).  The
fixtures are small (<1 MB) and committed; tests/test_oracle.py checks the
restatement in oracle/restate.py against them on any machine, and the GPU
parity tests check the CUDA path against them on the B200 box, where
/root/reference does not exist.  TEST INFRASTRUCTURE ONLY.
"""
import contextlib
import hashlib
import os

import numpy as np
import torch

from . import ref_harness, restate, synth

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

# strides chosen co-prime with the tensor extents so samples hit all channels/rows/cols
STRIDES = dict(logits=397, locs=1, w=1, image=251, fea64=4099, fea32=2053, sr=1021)
# denser samples (~15k values per output) for the module-level pin
MODULE_STRIDES = dict(logits=31, locs=1, w=1, image=7, fea64=127, fea32=67, sr=53)


def sample(t, stride):
    return t.detach().reshape(-1)[::stride].double().numpy().astype(np.float32)


def sd_digest(sd):
    h = hashlib.sha256()
    for k in sd:
        h.update(k.encode())
        h.update(sd[k].contiguous().numpy().tobytes())
    return h.hexdigest()


def case_inputs(name):
    """Seeded inputs of the golden cases (shared with the tests)."""
    if name == "config2":       # SURVEY.md section 8d config 2: B=1 line, 16 chars, regular grid
        return dict(lq=synth.make_lq(1, 0), labels=[synth.make_labels(16, 0)], locs=synth.make_locs(1, 16))
    if name == "ragged":        # clipped / overlapping windows, 5 chars, B=2 lines (3 + 2 chars)
        locs = synth.make_locs(2, 3, ragged=True, seed=7)
        locs[1, 4:] = 0
        locs[1, 0] = 250.2 / 512.0
        locs[1, 2] = 262.9 / 512.0  # overlaps the previous window: last writer wins
        return dict(lq=synth.make_lq(2, 10), labels=[synth.make_labels(3, 1), synth.make_labels(2, 2)], locs=locs)
    raise KeyError(name)


def run_reference(models, inp):
    lq, labels, locs = inp["lq"], inp["labels"], inp["locs"]
    with torch.no_grad():
        logits, enc_locs, w = models["encoder"](lq)
        imgs, p64, p32 = [], [], []
        for b in range(lq.shape[0]):
            img, f64, f32_ = models["tspgan"](styles=w[b:b + 1].repeat(labels[b].shape[0], 1), labels=labels[b], noise=None)
            imgs.append(img); p64.append(f64); p32.append(f32_)
        sr = models["sr"](lq, p64, p32, locs)
    return dict(logits=logits, enc_locs=enc_locs, w=w, image=torch.cat(imgs), fea64=torch.cat(p64),
                fea32=torch.cat(p32), sr=sr)


# CPU threads the golden fixtures were generated with.  The CPU convolutions split their sums by thread count, so the
# exact comparisons with them run with the same count whatever the host has.
GOLDEN_THREADS = 8


@contextlib.contextmanager
def golden_threads():
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    try:
        yield
    finally:
        torch.set_num_threads(n)


def modules_case():
    """Inputs of the module-level pin (tests/test_oracle.py::test_oracle_is_bit_identical_to_reference_modules)."""
    return synth.make_lq(1, 5), synth.make_labels(2, 9), synth.make_locs(1, 2, ragged=True, seed=3)


def write_modules_golden():
    """tests/golden/modules.npz: samples of every output of the three reference modules for modules_case(), with the
    reference's own w feeding TSPGAN and its own priors feeding TSPSRNet; w and the encoder locations are stored whole."""
    sds = synth.make_checkpoints(0)
    with golden_threads():
        lq, labels, locs = modules_case()
        ref = ref_harness.build_reference_models(sds)
        with torch.no_grad():
            rl, rlo, rw = ref["encoder"](lq)
            ri, r64, r32 = ref["tspgan"](styles=rw.repeat(2, 1), labels=labels, noise=None)
            rs = ref["sr"](lq, [r64], [r32], locs)
    out = dict(logits=rl, locs=rlo, w=rw, image=ri, fea64=r64, fea32=r32, sr=rs)
    rec = {k: sample(v, MODULE_STRIDES[k]) for k, v in out.items()}
    np.savez_compressed(os.path.join(GOLDEN_DIR, "modules.npz"), **rec)
    print("modules", {k: v.shape for k, v in rec.items()})


def main():
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    write_modules_golden()
    sds = synth.make_checkpoints(0)
    models = ref_harness.build_reference_models(sds)   # strict=True load == key/shape contract
    meta = {k: sd_digest(v) for k, v in sds.items()}
    for name in ("config2", "ragged"):
        inp = case_inputs(name)
        with golden_threads():
            out = run_reference(models, inp)
        rec = dict(
            logits=sample(out["logits"], STRIDES["logits"]), locs=sample(out["enc_locs"], 1), w=sample(out["w"], 1),
            image=sample(out["image"], STRIDES["image"]), fea64=sample(out["fea64"], STRIDES["fea64"]),
            fea32=sample(out["fea32"], STRIDES["fea32"]), sr=sample(out["sr"], STRIDES["sr"]),
            argmax=out["logits"].argmax(-1).numpy().astype(np.int64),
            sum_sr=np.float64(out["sr"].double().sum().item()), sum_image=np.float64(out["image"].double().sum().item()),
        )
        # window integers exactly as the reference computes them (networks.py:426-441, 460-474)
        wins = []
        for b in range(inp["lq"].shape[0]):
            for c in range(inp["labels"][b].shape[0]):
                wins.append(restate.char_window(inp["locs"][b][2 * c], 512, 16) + restate.char_window(inp["locs"][b][2 * c], 1024, 32))
        rec["windows"] = np.asarray(wins, dtype=np.int64)
        np.savez_compressed(os.path.join(GOLDEN_DIR, f"{name}.npz"), **rec)
        print(name, {k: (v.shape if hasattr(v, "shape") else v) for k, v in rec.items()})
    with open(os.path.join(GOLDEN_DIR, "checkpoint_sha256.txt"), "w") as f:
        for k, v in meta.items():
            f.write(f"{k} {v}\n")
    print(meta)


if __name__ == "__main__":
    main()

"""The reference's UNMODIFIED caller scripts against this repo's drop-in `models` package (SURVEY.md section 8b).

Reference sources are never committed: `build()` copies the scripts, utils/ and models/ into the git-ignored `oracle/_ref/`
when the reference tree is readable (oracle/stage_ref.py), and every test here skips when that copy is absent.  The copies
are verified against the committed SHA-256 list, so what runs IS the reference script.  Two settings:
* CPU (`reference` marker): test_sr.py against the reference's own models on the CPU (BASELINE configs[0]: plumbing,
  proves the harness and stubs), and against the drop-in, which must get through construction, strict checkpoint load,
  .eval(), .to(device), the parameter banner, and then fail LOUDLY at the first forward (there is no CPU fallback);
* GPU (`gpu` marker): `test_sr.py` and `test_w.py` run to completion on the B200 implementation, and the written PNGs are
  compared with the goldens the same scripts produced with the reference's own models on the CPU
  (`oracle/make_golden_script.py`, `oracle/make_golden_script_w.py`): within one grey level.
"""
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STUBS = os.path.join(ROOT, "oracle", "stubs")
STAGED = os.path.join(ROOT, "oracle", "_ref")
GOLDEN = os.path.join(ROOT, "tests", "golden")
BANNERS = ("43.062275 M Parameters", "27.970194 M Parameters", "16.865923 M Parameters")


def _write_checkpoints(d, checkpoints):
    os.makedirs(os.path.join(d, "checkpoints"), exist_ok=True)
    for key, name in (("tspgan", "net_prior_generation.pth"), ("sr", "net_sr.pth"), ("encoder", "net_transformer_encoder.pth")):
        torch.save({"params": checkpoints[key]}, os.path.join(d, "checkpoints", name))


def _write_line_image(d):
    import cv2
    os.makedirs(os.path.join(d, "LQs"), exist_ok=True)
    img = np.random.default_rng(0).integers(0, 256, (32, 256, 3), dtype=np.uint8)    # the image of oracle/make_golden_script.py
    cv2.imwrite(os.path.join(d, "LQs", "line0.png"), img)


def _run(cwd, script, pythonpath, args, timeout=900):
    env = dict(os.environ, PYTHONPATH=os.pathsep.join(pythonpath), OMP_NUM_THREADS=str(os.cpu_count() or 1), OPENCV_IPP="disabled")
    return subprocess.run([sys.executable, script] + args, cwd=cwd, env=env, capture_output=True, text=True, timeout=timeout)


def _require_staged():
    if not os.path.isfile(os.path.join(STAGED, "test_sr.py")):
        pytest.skip("oracle/_ref/ absent: build() stages it only where the reference tree is readable")


def _swapped_layout(d):
    """A user swaps the reference's models/ directory for dropin/models.  Python puts the script's own directory first on
    sys.path, so to emulate that checkout the byte-identical scripts are copied (at test time, into the temp dir only) next
    to a symlink of the reference's utils/ -- the reference's models/ is then NOT importable from this layout."""
    import shutil
    os.makedirs(d / "swapped")
    for script in ("test_sr.py", "test_w.py"):
        shutil.copy(os.path.join(STAGED, script), d / "swapped" / script)
    os.symlink(os.path.join(STAGED, "utils"), d / "swapped" / "utils")


# ------------------------------------------------------------------------------------------ CPU (reference's own models)
@pytest.fixture(scope="module")
def workdir(tmp_path_factory, checkpoints):
    _require_staged()
    d = tmp_path_factory.mktemp("marconet_run")
    _write_checkpoints(d, checkpoints)
    _write_line_image(d)
    _swapped_layout(d)
    return d


@pytest.mark.reference
def test_reference_script_with_reference_models_cpu(workdir):
    r = _run(workdir, os.path.join(STAGED, "test_sr.py"), [STUBS], ["-i", "./LQs", "-o", "./out_ref"])
    assert r.returncode == 0, r.stderr[-2000:]
    assert all(b in r.stdout for b in BANNERS)
    assert len(os.listdir(workdir / "out_ref")) == 1


@pytest.mark.reference
def test_reference_script_with_dropin_models(workdir):
    import filecmp
    assert filecmp.cmp(workdir / "swapped" / "test_sr.py", os.path.join(STAGED, "test_sr.py"), shallow=False)
    r = _run(workdir, str(workdir / "swapped" / "test_sr.py"), [os.path.join(ROOT, "dropin"), ROOT, STUBS], ["-i", "./LQs", "-o", "./out_b200"])
    # identical banner = identical parameter sets, after construction + strict load from ./checkpoints/*.pth
    assert all(b in r.stdout for b in BANNERS), r.stdout[-1500:] + r.stderr[-1500:]
    if torch.cuda.is_available():
        assert r.returncode == 0, r.stderr[-2000:]
        assert len(os.listdir(workdir / "out_b200")) == 1
    else:
        assert r.returncode != 0 and "no CPU fallback" in r.stderr, r.stderr[-1500:]


@pytest.mark.reference
def test_staged_hash_list_matches_reference():
    """The committed hash list (what the GPU test trusts) describes the staged reference files."""
    _require_staged()
    for line in open(os.path.join(GOLDEN, "reference_scripts_sha256.txt")).read().splitlines():
        digest, rel = line.split()
        assert hashlib.sha256(open(os.path.join(STAGED, rel), "rb").read()).hexdigest() == digest, rel


# ------------------------------------------------------------------------------------------ GPU (staged byte-identical copies)
@pytest.fixture(scope="module")
def staged(tmp_path_factory, checkpoints):
    _require_staged()
    for line in open(os.path.join(GOLDEN, "reference_scripts_sha256.txt")).read().splitlines():
        digest, rel = line.split()
        got = hashlib.sha256(open(os.path.join(STAGED, rel), "rb").read()).hexdigest()
        assert got == digest, f"{rel}: staged copy is not the reference file"
    d = tmp_path_factory.mktemp("marconet_gpu_run")
    _write_checkpoints(d, checkpoints)
    _write_line_image(d)
    _swapped_layout(d)
    return d


@pytest.mark.gpu
def test_unmodified_test_sr_runs_on_b200_and_matches_reference_png(staged):
    """reference test_sr.py:39-232 byte-unmodified, `models` = dropin/models (this repo's kernels), on the GPU."""
    import cv2
    r = _run(staged, str(staged / "swapped" / "test_sr.py"), [os.path.join(ROOT, "dropin"), ROOT, STUBS], ["-i", "./LQs", "-o", "./out_b200"])
    assert r.returncode == 0, r.stderr[-3000:]
    assert all(b in r.stdout for b in BANNERS), r.stdout[-1500:]
    outs = os.listdir(staged / "out_b200")
    assert len(outs) == 1, outs
    png = cv2.imread(str(staged / "out_b200" / outs[0]))
    assert png is not None and png.shape[0] == 4 * 128, None if png is None else png.shape
    g = np.load(os.path.join(GOLDEN, "script_sr_row.npz"))
    stride = int(g["stride"])
    sr_row = png[256:384][::stride, ::stride].astype(np.int64)        # rows: ShowLQ, ShowLocs, ShowSR, prior (test_sr.py:231)
    ref = g["sr_row"].astype(np.int64)
    assert sr_row.shape == ref.shape
    diff = np.abs(sr_row - ref)
    print("test_sr.py on B200 vs reference PNG: max grey-level diff", diff.max(), "pixels differing", int((diff > 0).sum()), "of", diff.size)
    assert diff.max() <= 1


@pytest.mark.gpu
def test_unmodified_test_w_runs_on_b200_and_matches_reference_pngs(staged):
    """reference test_w.py:42-117 byte-unmodified (11 interpolation PNGs + GIF) on the GPU implementation."""
    import cv2
    from oracle.make_golden_script_w import make_inputs
    gpath = os.path.join(GOLDEN, "script_w.npz")
    if not os.path.isfile(gpath):
        pytest.skip("tests/golden/script_w.npz not generated")
    make_inputs(str(staged / "in"))
    r = _run(staged, str(staged / "swapped" / "test_w.py"), [os.path.join(ROOT, "dropin"), ROOT, STUBS],
             ["-w1", "./in/w1.png", "-w2", "./in/w2.png", "-o", "./out_w"])
    assert r.returncode == 0, r.stderr[-3000:]
    assert "Finishing interpolation." in r.stdout
    assert os.path.isfile(staged / "out_w" / "w.gif")
    g = np.load(gpath)
    sy, sx = int(g["sy"]), int(g["sx"])
    worst = 0
    for i in range(11):
        png = cv2.imread(str(staged / "out_w" / "w_{:.2f}.png".format(i / 10)))
        assert png is not None and png.shape[1] == int(g["width"]), "character count differs from the reference run (argmax labels)"
        diff = np.abs(png[::sy, ::sx].astype(np.int64) - g[f"png{i}"].astype(np.int64))
        worst = max(worst, int(diff.max()))
    print("test_w.py on B200 vs reference PNGs: max grey-level diff", worst)
    assert worst <= 1

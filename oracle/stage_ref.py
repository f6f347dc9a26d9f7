"""Copy the reference's caller scripts and modules into the git-ignored oracle/_ref/ (TEST INFRASTRUCTURE ONLY).

The drop-in contract (SURVEY.md section 8b) is that the reference's `test_sr.py` / `test_w.py` run BYTE-UNMODIFIED with
`dropin/models` providing `models`.  Reference sources are never committed, so `build()` stages them here whenever the
reference tree is readable; the staged tree travels with the built package to a GPU machine, where
`tests/test_dropin_scripts.py` runs the scripts.  Every staged script is checked against the committed
`tests/golden/reference_scripts_sha256.txt`, so what the tests run is the unmodified reference file.

    python -m oracle.stage_ref                   # stage (a no-op when the reference tree is not readable)
    python -m oracle.stage_ref --write-hashes    # (re)generate the committed hash list from the reference tree
"""
import hashlib
import os
import shutil
import sys

from .ref_harness import REFERENCE_ROOT

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DST = os.path.join(ROOT, "oracle", "_ref")
HASHES = os.path.join(ROOT, "tests", "golden", "reference_scripts_sha256.txt")
SCRIPTS = ["test_sr.py", "test_w.py", "utils/alphabets.py", "utils/yolo_ocr_xloc.py"]
MODELS = ["models/networks.py", "models/ocr.py", "models/resnet.py", "models/textvit_arch.py"]


def sha(path):
    with open(path, "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()


def available():
    return all(os.access(os.path.join(REFERENCE_ROOT, rel), os.R_OK) for rel in SCRIPTS + MODELS)


def stage():
    """Copies SCRIPTS + MODELS to oracle/_ref/ and returns its path, or returns None when the reference tree is not readable.
    Raises when a script differs from the committed hash list."""
    if not available():
        return None
    want = dict(line.split()[::-1] for line in open(HASHES).read().splitlines() if line.strip())
    shutil.rmtree(DST, ignore_errors=True)
    for rel in SCRIPTS + MODELS:
        os.makedirs(os.path.dirname(os.path.join(DST, rel)), exist_ok=True)
        shutil.copyfile(os.path.join(REFERENCE_ROOT, rel), os.path.join(DST, rel))
    for rel in SCRIPTS:
        if sha(os.path.join(DST, rel)) != want[rel]:
            raise RuntimeError(f"{rel}: the reference file differs from {HASHES}")
    return DST


def main():
    if "--write-hashes" in sys.argv:
        if not available():
            raise SystemExit(f"reference tree not readable at {REFERENCE_ROOT}")
        with open(HASHES, "w") as f:
            for rel in SCRIPTS:
                f.write(f"{sha(os.path.join(REFERENCE_ROOT, rel))}  {rel}\n")
        print("wrote", HASHES)
    print("staged ->", stage())


if __name__ == "__main__":
    main()

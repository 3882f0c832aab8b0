"""BASELINE INFRASTRUCTURE ONLY — stages the UNMODIFIED reference (ultralytics/yolov3 @ 97b87b1) under the git-ignored
``oracle/_ref/`` when a checkout of it is at hand, so that a built tree carries it to machines that have none.  Nothing
under ``yolov3_b200/`` and no test imports it; the only consumers are ``bench.py --impl reference`` / ``bench.py``'s
``cpu_baseline`` leg (the reference's own ``Model`` / ``non_max_suppression`` timed on the host cores) and its
``gpu_library_baseline`` leg.  Without it they fall back to the oracle port or report themselves unavailable.

Why a file copy and not ``pip install --target``: the reference's pyproject.toml declares no ``version`` (setuptools:
"`project` must contain ['version'] properties") and its layout is a flat script tree (``models/``, ``utils/``,
``detect.py`` at top level: not an installable distribution), so metadata generation fails before anything is built.  The
reference is meant to be run from a clone (its README); a clone of the needed files is what this makes.  Files are copied
byte for byte, never edited; ``oracle/_ref/`` is listed in .gitignore so no reference source enters this repository.

    python oracle/stage_reference.py            # no-op when no reference checkout is present or it is already staged
"""
from __future__ import annotations

import shutil
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
SRC = Path("/root/reference")
DST = ROOT / "oracle" / "_ref"
# what the hot path's callers import: the model/graph code, the utils they pull in, the three loop scripts, YAMLs, the two
# sample images of BASELINE config 1 and the hyper-parameter files ComputeLoss reads
TOP_FILES = ["detect.py", "val.py", "train.py", "hubconf.py", "export.py", "LICENSE"]
TREES = ["models", "utils", "data/hyps", "data/images"]
DATA_FILES = ["data/coco128.yaml", "data/coco.yaml"]


def staged() -> bool:
    return (DST / "models" / "yolo.py").exists()


def source_available() -> bool:
    try:
        return (SRC / "models" / "yolo.py").exists()
    except OSError:  # a checkout the building user may not read: nothing to stage
        return False


def stage(force: bool = False) -> Path | None:
    if not source_available():
        return DST if staged() else None
    if staged() and not force:
        return DST
    if DST.exists():
        shutil.rmtree(DST)
    DST.mkdir(parents=True)
    ignore = shutil.ignore_patterns("__pycache__", "*.pyc", "*.ipynb", "docker", "aws", "google_app_engine", "flask_rest_api")
    for t in TREES:
        if (SRC / t).exists():
            shutil.copytree(SRC / t, DST / t, ignore=ignore)
    for f in TOP_FILES + DATA_FILES:
        if (SRC / f).exists():
            (DST / f).parent.mkdir(parents=True, exist_ok=True)
            shutil.copy2(SRC / f, DST / f)
    (DST / "STAGED_FROM").write_text(f"{SRC} (ultralytics/yolov3 @ 97b87b1), byte-for-byte copy by oracle/stage_reference.py\n")
    return DST


if __name__ == "__main__":
    p = stage(force="--force" in sys.argv)
    print(p if p else "reference not available here and nothing staged")

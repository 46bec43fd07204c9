#!/usr/bin/env python
"""Copy the few reference files the timing arm needs into the git-ignored ``baseline/_ref/`` -- TEST/BENCH INFRASTRUCTURE.

    python oracle/fetch_reference.py            # no-op when /root/reference is absent (the GPU box)

``/root/reference`` does not exist on the GPU box, but ``bench.py --impl reference`` must time the reference AS WRITTEN
there (SURVEY.md section 8c "GPU box caveat", VERDICT r01 item 6).  ``baseline/_ref/`` is listed in ``.gitignore`` (the
reference's sources never enter this repository's history) but not in ``.gpurunignore``, so the copy travels with the
snapshot exactly like the built ``.so``.  Only the files ``src/main.py`` imports on the hot path are copied, unmodified.
Run it by hand where the checkout is present; the build does not depend on it.
"""
from __future__ import annotations

import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.environ.get("HIPAC_REFERENCE_SRC", "/root/reference")
DST = os.path.join(ROOT, "baseline", "_ref")
FILES = [
    "src/__init__.py", "src/main.py",
    "src/models/__init__.py", "src/models/resnet.py", "src/models/simclr.py",
    "src/datasets/patch_dataset.py", "src/datasets/simclr_dataset.py",
    "src/utils/__init__.py", "src/utils/evaluation_FROC.py",
]


def fetch(verbose: bool = False) -> bool:
    """Returns True when ``baseline/_ref`` holds a usable copy afterwards."""
    if os.path.isfile(os.path.join(SRC, "src", "main.py")):
        for rel in FILES:
            s, d = os.path.join(SRC, rel), os.path.join(DST, rel)
            if not os.path.isfile(s):
                continue
            os.makedirs(os.path.dirname(d), exist_ok=True)
            if not os.path.exists(d) or os.path.getmtime(s) > os.path.getmtime(d) or os.path.getsize(s) != os.path.getsize(d):
                shutil.copyfile(s, d)
                if verbose:
                    print("copied", rel)
    return os.path.isfile(os.path.join(DST, "src", "main.py"))


if __name__ == "__main__":
    ok = fetch(verbose=True)
    print("baseline/_ref", "ready" if ok else "absent (no reference checkout here)")
    sys.exit(0)

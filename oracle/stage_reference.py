"""Stage the UNMODIFIED original ST-MGCN project under ``oracle/_ref/``.  TEST INFRASTRUCTURE.

    python oracle/stage_reference.py <checkout of underdoc-wang/ST-MGCN>

``__graft_entry__.build()`` does the same with the first checkout ``find_original()`` finds.  Copies its five
MIT-licensed Python files and its licence, byte for byte, into ``oracle/_ref/``.  The directory is git-ignored: the
original sources never enter this repository's history.  What reads it, when it is there:

* ``oracle/make_golden.py``, which runs the original modules to write the fixtures under ``tests/golden/``;
* ``tests/test_gpu_dropin_main.py``, which runs the original ``Main.py`` / ``Model_Trainer.py`` on this repository's
  drop-in modules (it skips when nothing is staged);
* ``bench.py``'s CPU baseline, which times the original modules (the oracle's restatement when nothing is staged).

No product module imports from there.
"""
from __future__ import annotations

import filecmp
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(HERE, "_ref")
REF_FILES = ("GCN.py", "STMGCN.py", "Model_Trainer.py", "Main.py", "Data_Container.py", "LICENSE")
# where build() looks for a checkout of the original: a directory named ``reference`` next to this repository, then
# ``/root/reference``, where the build containers of this project keep it
ORIGINAL_CANDIDATES = (os.path.join(os.path.dirname(HERE), "..", "reference"), "/root/reference")


def is_original(path: str) -> bool:
    return all(os.path.isfile(os.path.join(path, name)) and os.access(os.path.join(path, name), os.R_OK)
               for name in REF_FILES)


def find_original():
    """The first readable checkout of the original among ``ORIGINAL_CANDIDATES``, or None."""
    return next((os.path.abspath(p) for p in ORIGINAL_CANDIDATES if is_original(p)), None)


def stage(src: str) -> str:
    if not is_original(src):
        raise FileNotFoundError(f"{src} is not a readable checkout of the original ST-MGCN (needs {REF_FILES})")
    os.makedirs(REF_DIR, exist_ok=True)
    for name in REF_FILES:
        s, d = os.path.join(src, name), os.path.join(REF_DIR, name)
        if not (os.path.exists(d) and filecmp.cmp(s, d, shallow=False)):
            shutil.copyfile(s, d)
    return REF_DIR


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    print(f"staged {sys.argv[1]} -> {stage(sys.argv[1])}")

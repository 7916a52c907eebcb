#!/usr/bin/env python
"""Copy the UNMODIFIED reference files the tests / bench need from a checkout of the reference into baseline/_ref.

  python baseline/fetch_ref.py <reference checkout>

baseline/_ref is git-ignored (the reference's sources never enter the history):
  models/                         the reference's model classes  (bench.py --impl reference, live-oracle tests)
  speed_test.py, inference.py     the reference's entry points   (tests/test_zz_gpu_scripts.py runs them against the drop-in models/)
  data_handling/, tools/utils.py  what those two scripts import
The tests that need these files skip without them.
"""
import filecmp
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DST = os.path.join(HERE, "_ref")
FILES = ["speed_test.py", "inference.py", "data_handling/__init__.py", "data_handling/data_class.py", "tools/utils.py"]
MODEL_DIRS = ["WindowTransformer", "FastTransformer", "ResidualTransformer", "BicubicInterpolation"]


def fetch(ref: str, verbose: bool = False) -> bool:
    if not os.path.isdir(ref):
        return False
    files = list(FILES)
    for m in MODEL_DIRS:
        src = os.path.join(ref, "models", m)
        for f in os.listdir(src):
            if f.endswith(".py"):
                files.append(os.path.join("models", m, f))
    for rel in sorted(set(files)):
        s, d = os.path.join(ref, rel), os.path.join(DST, rel)
        os.makedirs(os.path.dirname(d), exist_ok=True)
        if not os.path.exists(d) or not filecmp.cmp(s, d, shallow=False):
            shutil.copyfile(s, d)
            if verbose:
                print("copied", rel)
    return True


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    print("fetched" if fetch(sys.argv[1], True) else f"no directory {sys.argv[1]}")

#!/usr/bin/env python
"""Golden vectors of the seeded ragged-shape sweep (tests/test_gpu_models.py::_ragged_cases), CPU, fp32.

  python tests/golden/make_ragged.py

Writes tests/golden/ragged_<k>.npz: the pre-clamp output of oracle.upscaler_oracle sampled by
tests/golden/cases.py::ragged_sample (a coprime-stride lattice plus dense crops of the four corners), and the case it belongs
to.  The reference's sources are not part of this repository: the stored values come from the oracle, whose arithmetic (oracle/upscaler_oracle.py) is the one that matched the UNMODIFIED reference
modules on every case of this sweep to 2e-5 when the sweep was added.  tests/test_oracle_golden.py checks the oracle against
these files, and against the reference itself whenever a copy of its models/ is in baseline/_ref.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import upscaler_oracle as orc                       # noqa: E402
from oracle.weights import synth_state_dict, synth_frames     # noqa: E402
from tests.golden.cases import RAGGED_CORNERS, ragged_sample  # noqa: E402
from tests.test_gpu_models import _ragged_cases               # noqa: E402


def main():
    for k, (model, shape, kw, seed) in enumerate(_ragged_cases()):
        B, H, W = shape
        sd = synth_state_dict(model, seed)
        x = synth_frames(B, H, W, seed=seed + 100)
        pre = orc.forward(model, sd, x, pre_clamp=True, **kw).numpy().astype(np.float32)
        st, lat, crops = ragged_sample(pre)
        out = dict(pre=lat, stride=st, shape=np.array(pre.shape), model=model, kw=repr(sorted(kw.items())), seed=seed)
        for i, cr in enumerate(crops):
            out[f"crop{i}"] = cr
        path = os.path.join(HERE, f"ragged_{k:02d}.npz")
        np.savez_compressed(path, **out)
        print(path, model, shape, kw, "stride", st, "corners", len(RAGGED_CORNERS), os.path.getsize(path), "bytes", flush=True)


if __name__ == "__main__":
    main()

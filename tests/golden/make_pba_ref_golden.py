"""Generates tests/golden/pba_ref_optimum.npz: what the reference's vendored PBA (lib/PBA, CPU double, built by oracle/Makefile
into oracle/_ref/libpba_ref.so) reaches on the bundle-adjustment problem of tests/test_pba_shim.py, driven by
oracle/pba_ref_shim.cc as the reference's ParallelBundleAdjuster::Solve() drives it.  The GPU test compares the same driver,
compiled against include/dagsfm_b200/pba_shim.hpp, with these numbers.  Run where the reference tree exists:
    make -C oracle ref && python tests/golden/make_pba_ref_golden.py"""
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

from oracle import pyoracle as orc  # noqa: E402
from tests.ba_scene import make_ba_problem  # noqa: E402
from tests.test_pba_shim import PROBLEM  # noqa: E402


def main():
    assert orc.pba_ref_available(), "build oracle/_ref first (make -C oracle ref, needs the reference tree)"
    r = orc.pba_ref_solve(make_ba_problem(**PROBLEM), max_iter=50)
    out = {k: np.asarray(r[k]) for k in ("initial_mse", "final_mse", "lm_iterations", "focal", "radial")}
    np.savez_compressed(ROOT / "tests" / "golden" / "pba_ref_optimum.npz", **out)
    print("written", {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()

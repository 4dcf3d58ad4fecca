"""SURVEY row B6: the PBA seam (ParallelBundleAdjuster, bundle_adjustment.cc:548-772).

oracle/pba_ref_shim.cc drives `pba::ParallelBA` exactly as the reference's Solve() does.  It is
compiled twice from the same source: against the reference's lib/PBA (oracle/_ref/libpba_ref.so,
the CPU reference) and against include/dagsfm_b200/pba_shim.hpp (b2_ba_solve on the GPU).  Both
must reach the same optimum; the reference's is stored in tests/golden/pba_ref_optimum.npz
(generator: tests/golden/make_pba_ref_golden.py)."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
DRV = ROOT / "tests" / "cpp" / "_pba_shim_drv.so"
PROBLEM = dict(n_img=24, n_pts=1500, track_len=6, seed=3, shared_camera=False)


def build():
    from dagsfm_b200 import build as b
    b.build()
    cmd = ["/usr/bin/g++", "-std=c++17", "-O1", "-shared", "-fPIC", "-DB2_PBA_SHIM", "-I", str(ROOT / "include"),
           str(ROOT / "oracle/pba_ref_shim.cc"), "-o", str(DRV), str(b.LIB), f"-Wl,-rpath,{b.LIB.parent}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return DRV


def test_pba_driver_compiles_against_the_shim():
    assert build().exists()


@pytest.mark.gpu
def test_pba_driver_reaches_the_reference_optimum_on_gpu():
    from oracle import pyoracle as orc
    from tests.ba_scene import make_ba_problem
    drv = DRV if DRV.exists() else build()
    g = orc.pba_ref_solve(make_ba_problem(**PROBLEM), max_iter=50, lib_path=drv)
    assert g["lm_iterations"] > 0 and g["final_mse"] < 0.25 * g["initial_mse"]
    r = np.load(ROOT / "tests" / "golden" / "pba_ref_optimum.npz")
    assert abs(g["initial_mse"] - r["initial_mse"]) <= 1e-4 * r["initial_mse"]
    # PBA stores float32 and stops on its own thresholds: same optimum to ~1e-3 relative
    assert abs(g["final_mse"] - r["final_mse"]) <= 2e-3 * r["final_mse"], (g["final_mse"], r["final_mse"])
    assert np.abs(g["focal"] - r["focal"]).max() < 1e-2 * np.abs(r["focal"]).max()

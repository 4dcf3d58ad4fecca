"""The matcher's host code and CUDA-core kernels (match_api.cu, match_post.cu, match_guided.cu) compiled for
the HOST against tests/cuda_emu/cuda_emu.h.  The two tcgen05 kernels have no CPU meaning; their place is
taken by tests/cuda_emu/match_tc_emu.cc, which produces what they are contracted to produce (best dot,
first 32-column chunk attaining it, best other-chunk maximum, candidate list).  Everything downstream --
items, fix-up (exact index + in-chunk second-best), cross-check, ordered compaction, chunking of long
pair lists, the two-slot seam, and the whole guided path -- is the real code, checked index-for-index
against the oracle.  TEST of the CUDA sources; the product library is not involved."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import pyoracle as orc
from tests.test_host_guided import _inlier_pairs, _scene_with_descriptors


@pytest.fixture(scope="module")
def mm():
    from tests.cuda_emu.build_emu import HERE, build
    import dagsfm_b200._lib as lm
    import dagsfm_b200.matching as mt
    L = C.CDLL(str(build("match", ["common.cu", "match_post.cu", "match_guided.cu", "match_api.cu"],
                         extra=[str(HERE / "match_tc_emu.cc")])))
    saved = (lm._lib, mt.check)
    lm._lib = None
    real_path = lm.LIB_PATH
    lm.LIB_PATH = type(real_path)(L._name)          # lib() binds the argtypes of the C ABI on the emulated library
    L2 = lm.lib()

    def check(rc):
        if rc != 0:
            raise RuntimeError(f"emulated library error {rc}: {L2.b2_last_error().decode()}")
    mt.check = check
    yield mt
    # the product library object comes back itself: the wrapper modules bound their argtypes on it once (a fresh CDLL
    # would leave e.g. bundle_adjustment's raw-pointer arguments unconverted, truncated to C ints)
    lm._lib, lm.LIB_PATH, mt.check = saved[0], real_path, saved[1]


def test_reference_cpu_vs_gpu_cases(mm):
    # sift_test.cc:496-557 through the two-slot seam (SetDescriptors / GetSiftMatch)
    gpu = mm.SiftMatchGPU(0)
    try:
        def both(o, d1, d2):
            exp = orc.match_sift(d1, d2, max_ratio=o.max_ratio, max_distance=o.max_distance, cross_check=o.cross_check)
            got = mm.match_sift_features_gpu(o, d1, d2, gpu)
            assert got.tolist() == exp.tolist()
            return len(exp)
        d1 = orc.create_random_descriptors(100)
        assert both(mm.SiftMatchingOptions(), d1, d1[::-1].copy()) == 100
        d2 = d1.copy()
        d2[99] = d2[0]
        r = d2[0].astype(np.float32); r[0] += 50.0; d2[0] = orc.l2_normalize_to_u8(r)
        r = d2[99].astype(np.float32); r[0] += 100.0; d2[99] = orc.l2_normalize_to_u8(r)
        assert both(mm.SiftMatchingOptions(max_ratio=0.4), d1[:99], d2) == 98
        assert both(mm.SiftMatchingOptions(max_ratio=0.5), d1, d2) == 99
        d1 = orc.create_random_descriptors(100); d2 = d1.copy(); d1[0] = d1[1]
        assert both(mm.SiftMatchingOptions(cross_check=False), d1, d2) == 100
        assert both(mm.SiftMatchingOptions(cross_check=True), d1, d2) == 98
        e = np.zeros((0, 128), np.uint8)
        assert len(mm.match_sift_features_gpu(mm.SiftMatchingOptions(), e, d2, gpu)) == 0
        # None keeps the previous upload of that slot (sift.h:232-234): slot 1 still holds d2
        assert mm.match_sift_features_gpu(mm.SiftMatchingOptions(), d1, None, gpu).tolist() == orc.match_sift(d1, d2).tolist()
    finally:
        gpu.close()



def test_no_cross_check_many_rows_few_columns_and_the_feature_clamp(mm):
    """ADVICE r1: without cross-check several rows of image 1 may share a column, so the match count can exceed n2 (the
    two-slot seam used to size its buffer by min(n1, n2) and fail); and the feature clamp of SiftMatchCU.cpp:108 --
    features beyond max_num_matches take no part -- holds on the two-slot AND the batched seam."""
    gpu = mm.SiftMatchGPU(0)
    try:
        d2 = orc.create_random_descriptors(40, seed=5)
        d1 = np.concatenate([d2, d2, d2, d2[:30]])          # 150 rows, every one an exact copy of a column of d2
        o = mm.SiftMatchingOptions(cross_check=False)
        exp = orc.match_sift(d1, d2, cross_check=False)
        assert len(exp) == 150 > len(d2)
        assert mm.match_sift_features_gpu(o, d1, d2, gpu).tolist() == exp.tolist()
        # clamp: only the first 100 / 25 features exist for the matcher
        oc = mm.SiftMatchingOptions(cross_check=False, max_num_matches=100)
        expc = orc.match_sift(d1[:100], d2, cross_check=False)
        assert mm.match_sift_features_gpu(oc, d1, d2, gpu).tolist() == expc.tolist()
        gpu.set_images([d1, d2])
        oc = mm.SiftMatchingOptions(cross_check=True, max_num_matches=25)
        off, m = gpu.match_pairs([(0, 1), (1, 0)], oc)
        assert m[off[0]:off[1]].tolist() == orc.match_sift(d1[:25], d2[:25]).tolist()
        assert m[off[1]:off[2]].tolist() == orc.match_sift(d2[:25], d1[:25]).tolist()
    finally:
        gpu.close()


def test_batched_pairs_ragged_and_chunked(mm, monkeypatch):
    monkeypatch.setenv("B2_MATCH_ROW_BUDGET", "65536")        # forces several chunks of pairs per call
    rng = np.random.default_rng(3)
    sizes = [300, 17, 0, 257, 64, 511]
    base = orc.create_random_descriptors(600, seed=4)
    descs = []
    for n in sizes:
        d = base[rng.permutation(600)[:n]].copy() if n else np.zeros((0, 128), np.uint8)
        descs.append(d)
    pairs = [(i, j) for i in range(len(sizes)) for j in range(len(sizes)) if i != j]
    gpu = mm.SiftMatchGPU(0)
    try:
        gpu.set_images(descs)
        for o in (mm.SiftMatchingOptions(), mm.SiftMatchingOptions(cross_check=False, max_ratio=0.95, max_distance=1.3)):
            off, m = gpu.match_pairs(pairs, o)
            for p, (i, j) in enumerate(pairs):
                exp = orc.match_sift(descs[i], descs[j], max_ratio=o.max_ratio, max_distance=o.max_distance,
                                     cross_check=o.cross_check)
                assert m[off[p]:off[p + 1]].tolist() == exp.tolist(), (p, i, j)
        with pytest.raises(RuntimeError):
            gpu.match_pairs([(0, 99)], mm.SiftMatchingOptions())
    finally:
        gpu.close()


def test_ties_and_duplicates(mm):
    d = orc.create_random_descriptors(40, seed=9)
    a = np.r_[d, d[:5]]                  # duplicated rows: ties for best -> the lowest index wins, ratio test fails
    b = np.r_[d[::-1], d[:3]].copy()
    gpu = mm.SiftMatchGPU(0)
    try:
        gpu.set_images([a, b])
        for cc in (True, False):
            o = mm.SiftMatchingOptions(cross_check=cc)
            off, m = gpu.match_pairs([(0, 1), (1, 0)], o)
            assert m[off[0]:off[1]].tolist() == orc.match_sift(a, b, cross_check=cc).tolist()
            assert m[off[1]:off[2]].tolist() == orc.match_sift(b, a, cross_check=cc).tolist()
    finally:
        gpu.close()


def test_guided_pairs_through_the_c_abi(mm):
    rng = np.random.default_rng(11)
    kps, descs, pairs, geos = [], [], [], []
    for k in range(4):
        planar = k % 2 == 1
        k1, k2, d1, d2 = _scene_with_descriptors(rng, 150 + 60 * k, 60 + 30 * k, planar)
        a, b = _inlier_pairs(k1, k2, d1, d2)
        geos.append((4 + k, None, orc.h_dlt(a, b)) if planar else (2 + k // 2, orc.eight_point(a, b), None))
        kps += [k1, k2]; descs += [d1, d2]; pairs.append((2 * k, 2 * k + 1))
    pairs += [(0, 1), (3, 2)]
    geos += [(0, None, None), geos[1]]
    gpu = mm.SiftMatchGPU(0)
    try:
        gpu.set_images(descs)
        with pytest.raises(RuntimeError):                      # keypoints are mandatory for the guided path
            gpu.match_guided_pairs(pairs, geos, mm.SiftMatchingOptions())
        with pytest.raises(RuntimeError):                      # and must match the descriptor counts (sift.cc:82-87)
            gpu.set_keypoints([k[:-1] for k in kps])
        gpu.set_keypoints(kps)
        for o in (mm.SiftMatchingOptions(), mm.SiftMatchingOptions(cross_check=False, max_error=2.0)):
            off, m = gpu.match_guided_pairs(pairs, geos, o)
            for p, ((i, j), (cfg, F, H)) in enumerate(zip(pairs, geos)):
                e = orc.match_guided(kps[i], kps[j], descs[i], descs[j], cfg, F=F, H=H, max_error=o.max_error,
                                     max_ratio=o.max_ratio, max_distance=o.max_distance, cross_check=o.cross_check)
                assert m[off[p]:off[p + 1]].tolist() == ([] if e is None else e.tolist()), (p, cfg)
        # guided and unguided share the object: the plain matcher still works afterwards
        off2, m2 = gpu.match_pairs(pairs[:1], mm.SiftMatchingOptions())
        assert m2[off2[0]:off2[1]].tolist() == orc.match_sift(descs[0], descs[1]).tolist()
        one = mm.match_guided_sift_features_gpu(mm.SiftMatchingOptions(), kps[0], kps[1], descs[0], descs[1], gpu,
                                                geos[0][0], F=geos[0][1])
        assert one.tolist() == orc.match_guided(kps[0], kps[1], descs[0], descs[1], geos[0][0], F=geos[0][1]).tolist()
    finally:
        gpu.close()


def test_pair_naming_an_unknown_image_is_rejected_without_touching_memory(mm):
    """A pair that references an image outside the store must come back as an error.  fill_items_kernel used to
    index img_n / img_row with the bad id (found by the emulator's guard pages; on the GPU it read whatever
    followed the allocation and could emit items for it)."""
    d = orc.create_random_descriptors(40, seed=2)
    gpu = mm.SiftMatchGPU(0)
    try:
        gpu.set_images([d, d[::-1].copy()])
        for bad in ([(0, 2)], [(7, 1)], [(0, 1), (1, 4000000000)]):
            with pytest.raises(RuntimeError):
                gpu.match_pairs(bad, mm.SiftMatchingOptions())
        off, m = gpu.match_pairs([(0, 1)], mm.SiftMatchingOptions())       # the handle stays usable
        assert m[off[0]:off[1]].tolist() == orc.match_sift(d, d[::-1].copy()).tolist()
    finally:
        gpu.close()


def test_saturating_and_zero_descriptors(mm):
    hi = np.full((70, 128), 255, np.uint8)          # every dot = 128 * 255^2: clamped distance, everything ties
    zero = np.zeros((33, 128), np.uint8)            # dots 0: no match at all (sift.cc:136-138)
    mix = np.r_[orc.create_random_descriptors(50, seed=3), zero[:5], hi[:2]]
    gpu = mm.SiftMatchGPU(0)
    try:
        gpu.set_images([hi, zero, mix])
        pairs = [(0, 0), (0, 1), (1, 1), (2, 2), (2, 0), (1, 2)]
        for o in (mm.SiftMatchingOptions(), mm.SiftMatchingOptions(cross_check=False, max_ratio=1.0, max_distance=1.5707964)):
            off, m = gpu.match_pairs(pairs, o)
            ds = [hi, zero, mix]
            for p, (i, j) in enumerate(pairs):
                exp = orc.match_sift(ds[i], ds[j], max_ratio=o.max_ratio, max_distance=o.max_distance, cross_check=o.cross_check)
                assert m[off[p]:off[p + 1]].tolist() == exp.tolist(), (p, i, j)
    finally:
        gpu.close()


def test_guided_cpp_shim_on_the_emulated_library():
    """include/dagsfm_b200/colmap_shim.hpp: the reference's TestMatchGuidedSiftFeaturesGPU replayed through
    MatchGuidedSiftFeaturesGPU, and the SiftMatchGPU guided interface (factory, SetFeautreLocation, GetGuidedSiftMatch)
    driven directly -- the C++ test program of tests/test_zz_guided_gpu.py linked against the emulated library."""
    import subprocess
    from pathlib import Path
    from tests.cuda_emu.build_emu import HERE, build
    root = Path(__file__).resolve().parent.parent
    lib = build("match", ["common.cu", "match_post.cu", "match_guided.cu", "match_api.cu"], extra=[str(HERE / "match_tc_emu.cc")])
    exe = HERE / "_build" / "guided_shim_test_emu"
    r = subprocess.run(["/usr/bin/g++", "-std=c++17", "-O1", "-I", str(root / "include"), str(root / "tests/cpp/guided_shim_test.cc"),
                        "-o", str(exe), str(lib), f"-Wl,-rpath,{lib.parent}"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "guided shim ok" in r.stdout, r.stdout + r.stderr


def test_matcher_cpp_shim_on_the_emulated_library():
    """The SiftMatchGPU / CreateSiftGPUMatcher / MatchSiftFeaturesGPU adaptors (tests/cpp/shim_test.cc, the reference's
    sift_test.cc cases) linked against the emulated library."""
    import subprocess
    from pathlib import Path
    from tests.cuda_emu.build_emu import HERE, build
    root = Path(__file__).resolve().parent.parent
    lib = build("match", ["common.cu", "match_post.cu", "match_guided.cu", "match_api.cu"], extra=[str(HERE / "match_tc_emu.cc")])
    exe = HERE / "_build" / "shim_test_emu"
    r = subprocess.run(["/usr/bin/g++", "-std=c++17", "-O1", "-I", str(root / "include"), str(root / "tests/cpp/shim_test.cc"),
                        "-o", str(exe), str(lib), f"-Wl,-rpath,{lib.parent}"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "shim ok" in r.stdout, r.stdout + r.stderr


def test_bench_guided_leg_runs_on_the_emulated_library(mm):
    """bench.py's opt-in guided-matching leg end to end on the emulated library (index-exact with the oracle)."""
    import sys
    import types
    argv, sys.argv = sys.argv, ["bench.py"]
    try:
        import bench
    finally:
        sys.argv = argv
    import dagsfm_b200
    saved = (dagsfm_b200.SiftMatchGPU, dagsfm_b200.SiftMatchingOptions)
    dagsfm_b200.SiftMatchGPU, dagsfm_b200.SiftMatchingOptions = mm.SiftMatchGPU, mm.SiftMatchingOptions
    try:
        out = bench.bench_guided(types.SimpleNamespace(guided_pairs=3), 0, 0, 1, 1, lambda: None)
    finally:
        dagsfm_b200.SiftMatchGPU, dagsfm_b200.SiftMatchingOptions = saved
    assert out["pairs"] == 3 and out["identical_to_oracle"] == "3/3" and out["matches_per_pair"] > 1000


def test_guided_stage_chained_on_device_results(mm):
    """b2_match_guided_pairs_device: geometries come from b2_two_view_result records in device memory (host memory on the
    emulator); equal to the host-buffer call with the same geometries; pairs below min_num_inliers and configurations
    without a guided filter yield empty slices (GuidedSiftGPUFeatureMatcher::Run, matching.cc:508-512)."""
    from dagsfm_b200.verification import RESULT_DTYPE
    rng = np.random.default_rng(3)
    kps, descs, geos = [], [], []
    for k in range(4):
        k1, k2, d1, d2 = _scene_with_descriptors(rng, 120 + 30 * k, 40, planar=(k % 2 == 1))
        a, b = _inlier_pairs(k1, k2, d1, d2)
        geos.append((6, None, orc.h_dlt(a, b)) if k % 2 else (2, orc.eight_point(a, b), None))
        kps += [k1, k2]
        descs += [d1, d2]
    pairs = np.array([(0, 1), (2, 3), (4, 5), (6, 7), (0, 1), (2, 3)], np.uint32)
    res = np.zeros(6, RESULT_DTYPE)
    for p in range(6):
        cfg, F, H = geos[p % 4]
        res["config"][p], res["n_inliers"][p] = cfg, 50
        res["F"][p] = np.zeros(9) if F is None else F.ravel()
        res["H"][p] = np.zeros(9) if H is None else H.ravel()
    res["n_inliers"][4] = 14            # below the gate
    res["config"][5] = 7                # WATERMARK: no guided filter
    o = mm.SiftMatchingOptions()
    gpu = mm.SiftMatchGPU(0)
    try:
        gpu.set_images(descs)
        gpu.set_keypoints(kps)
        off_h, m_h = gpu.match_guided_pairs(pairs[:4], geos, o)
        cap = int(sum(len(descs[a]) for a, _ in pairs))
        off_d = np.zeros(7, np.int64)
        m_d = np.zeros((cap, 2), np.uint32)
        total = gpu.match_guided_pairs_device(6, pairs.ctypes.data, res.ctypes.data, 15, o, off_d.ctypes.data, m_d.ctypes.data, cap)
    finally:
        gpu.close()
    assert off_d[:5].tolist() == off_h.tolist() and m_d[:off_h[-1]].tolist() == m_h.tolist()
    assert off_d[5] == off_d[4] == off_d[6] == total and total > 300

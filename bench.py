#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (BASELINE.json metric: image pairs VERIFIED per second + BA iter/s).

Headline workload (BASELINE configs[2], SURVEY.md 8d "C3"): a synthetic sequence of 5000 images x 4096 SIFT keypoints
(dagsfm_b200/synthetic.py: one long 3-D scene, neighbouring images overlap), the 50 candidate pairs per image a
retrieval stage would hand over (248 725 pairs), every pair through descriptor matching (sift.cc:76-198) AND two-view
geometric verification (two_view_geometry.cc:292-489) -- the reference's SiftFeatureMatcher pipeline
(feature/matching.cc:610-839) -- with the match lists staying on the device.  One "step" = one pass over the whole
candidate list.  `value` = candidate pairs verified per second with the images resident in HBM; `e2e` = the same pass
with descriptors, keypoints and pairs coming from pinned host memory and results + match / inlier lists going back.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]
    python bench.py --impl reference ...     # the reference's CPU path (oracle port) on the host cores

Multi-GPU: ONE pair list, cut into contiguous (locality-ordered) ranges, one per rank; rank 0 gathers the results
inside the timed region -> "strong" scaling.  Extra legs in the same JSON line: `match` (C2: 1000 x 4096 exhaustive
matching, tcgen05 roofline), `ba` (C4: 500 cams / 100k pts / 1M obs), `ba_c5` with --ba-c5 (10k cams, ITERATIVE_SCHUR).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "image_pairs_verified_per_s"
UNIT = "pairs/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--seq-images", type=int, default=5000, help="C3 pipeline: images in the sequence")
    ap.add_argument("--seq-kp", type=int, default=4096,
                    help="C3 pipeline: keypoints (= descriptors) per image (SURVEY 8d C3: 5000 images x 4096 descriptors; round 2's GPU sessions 7-21 measured with 2048)")
    ap.add_argument("--seq-cand", type=int, default=50, help="C3 pipeline: candidate pairs per image")
    ap.add_argument("--images", type=int, default=1000, help="C2 match leg: images")
    ap.add_argument("--desc", type=int, default=4096, help="C2 match leg: descriptors per image")
    ap.add_argument("--pairs", type=int, default=131072, help="C2 match leg: pairs per step (0 = all 499 500; -1 = skip the leg)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="pairs in the CPU baseline sample (0 = 24 per core)")
    ap.add_argument("--verify-pairs", type=int, default=0, help="opt-in leg: stand-alone verification of pre-matched pairs")
    ap.add_argument("--ba", default="500,100000,10", help="BA leg: images,points,track (empty = skip)")
    ap.add_argument("--ba-c5", default="10000,2000000,10",
                    help="second BA leg, the C5 shape (BASELINE configs[4]: 10 k images / 2 M points / 20 M observations; the "
                         "reference's rule selects ITERATIVE_SCHUR above 1000 images); images,points,track (empty = skip)")
    ap.add_argument("--guided-pairs", type=int, default=0,
                    help="opt-in leg: guided matching (b2_match_guided_pairs, MatchGuidedSiftFeaturesGPU) on this many synthetic pairs")
    ap.add_argument("--verify-pose", action="store_true",
                    help="verification leg: also time b2_verify_relative_pose (EstimateWithRelativePose) on the verified pairs")
    ap.add_argument("--ba-solver", default="auto", choices=["auto", "exact", "iterative"],
                    help="BA leg: linear solver (auto = the reference's rule: ITERATIVE_SCHUR above 1000 images)")
    ap.add_argument("--retrieval-words", type=int, default=32768,
                    help="retrieval leg (candidate pairs from a vocabulary tree over the C3 collection): visual words; 0 = skip")
    ap.add_argument("--c1", action="store_true",
                    help="BASELINE configs[0] (the reference's CPU-runnable plumbing case): 100 images x 2048 descriptors, EXHAUSTIVE "
                         "pairs (4950), match + verify; the CPU leg runs the oracle port on ALL pairs and every result is compared")
    ap.add_argument("--chunk-pairs", type=int, default=65536,
                    help="pairs per b2_match_pairs_device -> b2_verify_pairs_device call (one launch group of the stage kernels)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the C3 results of the last step as DIR/<name>.npy (float64; a fixed, "
                         f"seeded sample of {DUMP_MAX_PAIRS} pairs when there are more) to compare two builds output for output")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the results of the b200 arm")
    return a


DUMP_MAX_PAIRS = 1 << 17      # 38 float64 values per pair: at most 40 MB in all


def dump_outputs(out_dir, results, pairs):
    """What a caller of the timed C3 step receives -- one RESULT_DTYPE row per candidate pair -- as one float64 .npy per
    field, with the pairs and their indices in the candidate list.  The inputs are seeded, so the same arguments give the
    same files on any build that computes the same thing."""
    n = len(results)
    idx = np.arange(n) if n <= DUMP_MAX_PAIRS else np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_PAIRS, replace=False))
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    np.save(d / "pair_index.npy", idx.astype(np.float64))
    np.save(d / "pairs.npy", pairs[idx].astype(np.float64))
    for f in results.dtype.names:
        np.save(d / f"{f}.npy", results[f][idx].astype(np.float64))


# --------------------------------------------------------------------- workload
def make_descriptors_torch(n_img, n_desc, seed, device):
    """Synthetic scene (SURVEY 8d): a global pool of scene points with base descriptors drawn
    by the reference's test recipe (sift_test.cc:243-253: U(0,1)^2, L2-normalise, round(512 x),
    saturate); image i sees a sliding window of n_desc/2 points (so neighbouring images
    overlap) with per-view noise N(0, 0.03) before normalisation; the other half of its
    slots are independent random descriptors.  Returns uint8 [n_img, n_desc, 128] on device."""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    half = n_desc // 2
    stride = max(half // 8, 1)
    pool_n = stride * n_img + half
    base = torch.rand((pool_n, 128), generator=g, device=device) ** 2
    base = base / base.norm(dim=1, keepdim=True)
    out = torch.empty((n_img, n_desc, 128), dtype=torch.uint8, device=device)
    for i in range(n_img):
        v = base[i * stride:i * stride + half] + 0.03 * torch.randn((half, 128), generator=g, device=device) / 5.06
        v = v.clamp_min(0)
        r = torch.rand((n_desc - half, 128), generator=g, device=device) ** 2
        d = torch.cat([v, r])
        d = d / d.norm(dim=1, keepdim=True)
        d = torch.round(512.0 * d).clamp(0, 255).to(torch.uint8)
        perm = torch.randperm(n_desc, generator=g, device=device)
        out[i] = d[perm]
    return out


def effective_cores() -> int:
    """Host threads the process may actually use: affinity mask capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = Path("/sys/fs/cgroup/cpu.max").read_text().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except Exception:
        try:
            q = int(Path("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read_text())
            per = int(Path("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read_text())
            if q > 0:
                n = max(1, min(n, int(q / per + 0.5)))
        except Exception:
            pass
    return n


def all_pairs(n_img, limit=0):
    i, j = np.triu_indices(n_img, k=1)
    p = np.stack([i, j], axis=1).astype(np.uint32)
    if limit and limit < len(p):
        p = p[:limit]
    return np.ascontiguousarray(p)


# ----------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names)
                   if any(len(r) > 2 + k and r[2 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------ CPU baseline
def cpu_reference(descs_host, pairs, n_sample, threads):
    """Times the oracle port of MatchSiftFeaturesCPU (reference sift.cc:76-198,810-822) on a
    uniform sample of the step's pairs, `threads` workers each matching one pair at a time
    (as the reference's num_threads SiftCPUFeatureMatcher workers, matching.cc:640-644)."""
    from oracle import pyoracle as orc
    rng = np.random.default_rng(0)
    idx = np.sort(rng.choice(len(pairs), size=min(n_sample, len(pairs)), replace=False))
    sample = pairs[idx]
    secs, counts, _ = orc.match_pairs_mt(descs_host, sample, n_threads=threads)
    return len(sample) / secs, secs, len(sample), counts, idx



def peaks_hbm():
    try:
        return json.loads((ROOT / "MEASURED_PEAKS.json").read_text()).get("hbm_gbs", 6650.0), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def verify_work_rates(res, match_offsets, kernel_s):
    """SURVEY 8(d) unit of the verification stage: hypothesis-match evaluations (33 flop Sampson for E / F,
    25 flop for H).  Lower bound from the trial counts the kernel reports: every trial scores at least one
    hypothesis against all M matches (the 7-point solver yields up to 3, the 5-point up to 10), LO and
    tie-breaking passes not counted."""
    m = np.diff(np.asarray(match_offsets, dtype=np.int64)).astype(np.float64)
    ef = (res["E_num_trials"].astype(np.float64) + res["F_num_trials"].astype(np.float64)) * m
    h = res["H_num_trials"].astype(np.float64) * m
    evals = float(ef.sum() + h.sum())
    flops = float(33.0 * ef.sum() + 25.0 * h.sum())
    return {"hypothesis_match_evals_per_s_min": evals / kernel_s, "fp64_gflops_min": flops / kernel_s / 1e9,
            "fp64_peak_note": "lower bound (>= 1 hypothesis per trial); FP64 vector peak not in MEASURED_PEAKS.json, "
                              "public B200 figure ~40 TFLOP/s",
            "trials_per_pair": {k: float(res[k + "_num_trials"].mean()) for k in ("E", "F", "H")}}


def bench_verify(a, local_rank, rank, world, cores, barrier):
    """Two-view verification throughput: b2_verify_pairs (host buffers in / out) on synthetic
    matched pairs; CPU baseline = oracle port of TwoViewGeometry::Estimate, `cores` workers."""
    from dagsfm_b200 import Camera, TwoViewGeometryVerifier, TwoViewOptions
    from dagsfm_b200.tv_scene import make_pairs
    w = make_pairs(a.verify_pairs, seed=7 + rank)
    n = len(w["pairs"])
    cams = [Camera.make(params=w["cam_params"], prior_focal=bool(p)) for p in w["prior"]]
    v = TwoViewGeometryVerifier(local_rank)
    v.set_images(cams, w["keypoints"])
    opt = TwoViewOptions.default()
    seeds = (np.arange(n) * 2654435761 % (2 ** 32)).astype(np.uint32)
    res, inl = v.verify_pairs(w["pairs"], w["match_offsets"], w["matches"], opt, seeds)   # warm-up
    barrier()
    t0 = time.perf_counter()
    res, inl = v.verify_pairs(w["pairs"], w["match_offsets"], w["matches"], opt, seeds)
    barrier()
    wall = time.perf_counter() - t0
    kern = v.last_kernel_seconds()
    out = {"pairs": n * world, "matches_per_pair": float(w["match_offsets"][-1] / n),
           "pairs_per_s_e2e": n * world / wall, "pairs_per_s_kernel": n * world / kern,
           "config_histogram": {int(k): int(c) for k, c in zip(*np.unique(res["config"], return_counts=True))},
           "inlier_recall": float((res["n_inliers"] >= 0.9 * w["n_inliers_true"]).mean()),
           "api": "b2_verify_pairs (host buffers)"}
    try:
        out["roofline"] = verify_work_rates(res, w["match_offsets"], kern)
    except Exception as e:   # a reporting extra must never cost the bench line
        out["roofline"] = {"error": repr(e)}
    if getattr(a, "verify_pose", False):   # opt-in: the pose kernel has not been validated on a GPU yet
        try:
            v.relative_pose(w["pairs"], w["match_offsets"], res, inl)      # warm-up
            barrier()
            t1 = time.perf_counter()
            poses = v.relative_pose(w["pairs"], w["match_offsets"], res, inl)
            barrier()
            dt = time.perf_counter() - t1
            posed = int((np.abs(poses["qvec"]).sum(1) > 0).sum())
            out["relative_pose"] = {"pairs_per_s_e2e": n * world / dt, "pairs_with_pose": posed * world,
                                    "median_tri_angle_deg": float(np.degrees(np.median(poses["tri_angle"][poses["tri_angle"] > 0]))) if posed else 0.0,
                                    "api": "b2_verify_relative_pose (host buffers)"}
        except Exception as e:
            out["relative_pose"] = {"error": repr(e)}
    if rank == 0 and not a.no_cpu:
        from oracle import pyoracle as orc
        import ctypes as C
        ns = min(n, max(64, 1000 * cores))   # ~10-15 s of host work at ~80 pairs/s per core
        ocams = (orc.OrcCamera * (2 * ns))(*[orc.make_camera(params=w["cam_params"], prior=bool(p)) for p in w["prior"][:2 * ns]])
        ptrs = (C.c_void_p * (2 * ns))(*[k.ctypes.data for k in w["keypoints"][:2 * ns]])
        oo = orc.tv_default_options()
        ores = (orc.OrcTvResult * ns)()
        off = np.ascontiguousarray(w["match_offsets"][:ns + 1])
        oinl = np.zeros((int(off[-1]), 2), np.uint32)
        with orc.solver_stack(1):   # the oracle in the kernel's operation order: identity, not an agreement rate
            secs = orc._tv().orc_two_view_pairs_mt2(C.cast(ocams, C.c_void_p), C.cast(ptrs, C.c_void_p),
                                                    w["pairs"].ctypes.data, ns, off.ctypes.data, w["matches"].ctypes.data,
                                                    C.byref(oo), seeds.ctypes.data, cores, C.cast(ores, C.c_void_p), oinl.ctypes.data)
        same = sum(int(ores[i].config == res["config"][i] and ores[i].n_inliers == res["n_inliers"][i] and
                       ores[i].E_trials == res["E_num_trials"][i] and ores[i].F_trials == res["F_num_trials"][i] and
                       ores[i].H_trials == res["H_num_trials"][i] and
                       np.array_equal(oinl[off[i]:off[i] + max(ores[i].n_inliers, 0)], inl[off[i]:off[i] + max(int(res["n_inliers"][i]), 0)]) and
                       all(np.array_equal(np.array(getattr(ores[i], m)[:]).view(np.uint64), res[m][i].view(np.uint64)) for m in "EFH"))
                   for i in range(ns))
        out["cpu_baseline"] = {"value": ns / secs, "unit": "pairs/s", "cores": cores, "kind": "port",
                               "sample": f"{ns} pairs, {secs:.1f} s, oracle port of TwoViewGeometry::Estimate (device-order solver stack)",
                               "identical_to_gpu": f"{same}/{ns}",
                               "identical_means": "configuration, inlier and trial counts, inlier match list, E / F / H bit for bit"}
    v.close()
    return out


def _np_eight_point(x, y):
    """Guiding F for the synthetic guided-matching input: plain normalised 8-point in numpy (input generation only)."""
    def norm(p):
        c = p.mean(0)
        s = np.sqrt(2.0) / np.sqrt(((p - c) ** 2).sum(1)).mean()
        T = np.array([[s, 0, -s * c[0]], [0, s, -s * c[1]], [0, 0, 1.0]])
        return np.c_[p, np.ones(len(p))] @ T.T, T
    a1, T1 = norm(np.asarray(x, float))
    a2, T2 = norm(np.asarray(y, float))
    A = np.einsum("ni,nj->nij", a2, a1).reshape(-1, 9)
    F = np.linalg.svd(A)[2][-1].reshape(3, 3)
    u, sv, vt = np.linalg.svd(F)
    F = T2.T @ (u @ np.diag([sv[0], sv[1], 0.0]) @ vt) @ T1
    return F / np.linalg.norm(F)


def _np_h_dlt(x, y):
    """Guiding H for the synthetic guided-matching input: plain DLT in numpy (input generation only)."""
    x, y = np.asarray(x, float), np.asarray(y, float)
    rows = []
    for (u, v), (s, t) in zip(x, y):
        rows.append([-u, -v, -1, 0, 0, 0, s * u, s * v, s])
        rows.append([0, 0, 0, -u, -v, -1, t * u, t * v, t])
    H = np.linalg.svd(np.array(rows))[2][-1].reshape(3, 3)
    return H / H[2, 2]


def bench_guided(a, local_rank, rank, world, cores, barrier):
    """Guided matching throughput (SURVEY row M5, off by default in the reference): pairs of synthetic images with
    matched keypoints, outliers and repeated-structure decoys; the guiding F / H are a numpy 8-point / DLT on the true
    inliers (input generation); parity = index-exact with the oracle's MatchGuidedSiftFeaturesCPU on a sample of the
    pairs (the oracle is only that checker)."""
    from dagsfm_b200 import SiftMatchGPU, SiftMatchingOptions
    from tests.test_host_guided import _inlier_pairs, _scene_with_descriptors
    rng = np.random.default_rng(11 + rank)
    n_scenes = min(a.guided_pairs, 16)                  # distinct image pairs; the pair list cycles over them
    kps, descs, geos = [], [], []
    for k in range(n_scenes):
        planar = k % 2 == 1
        k1, k2, d1, d2 = _scene_with_descriptors(rng, 1500, 548, planar)      # 2048 keypoints per image
        x, y = _inlier_pairs(k1, k2, d1, d2)
        geos.append((6, None, _np_h_dlt(x, y)) if planar else (3, _np_eight_point(x, y), None))
        kps += [k1, k2]
        descs += [d1, d2]
    pairs = [(2 * (p % n_scenes), 2 * (p % n_scenes) + 1) for p in range(a.guided_pairs)]
    geometries = [geos[p % n_scenes] for p in range(a.guided_pairs)]
    opt = SiftMatchingOptions()
    m = SiftMatchGPU(local_rank)
    try:
        m.set_images(descs)
        m.set_keypoints(kps)
        off, mt = m.match_guided_pairs(pairs, geometries, opt)            # warm-up
        barrier()
        t0 = time.perf_counter()
        off, mt = m.match_guided_pairs(pairs, geometries, opt)
        barrier()
        wall = time.perf_counter() - t0
    finally:
        m.close()
    from oracle import pyoracle as orc                 # checker only, outside the timed region
    same = 0
    for p in range(min(n_scenes, 4)):
        cfg, F, H = geometries[p]
        e = orc.match_guided(kps[2 * p], kps[2 * p + 1], descs[2 * p], descs[2 * p + 1], cfg, F=F, H=H)
        same += int(mt[off[p]:off[p + 1]].tolist() == e.tolist())
    return {"pairs": a.guided_pairs * world, "keypoints_per_image": 2048, "pairs_per_s_e2e": a.guided_pairs * world / wall,
            "matches_per_pair": float(off[-1] / max(a.guided_pairs, 1)), "identical_to_oracle": f"{same}/{min(n_scenes, 4)}",
            "api": "b2_match_guided_pairs (host buffers)"}


def _mean_reproj(prob):
    try:
        from dagsfm_b200.ba_scene import mean_reprojection_error
        return mean_reprojection_error(prob)
    except Exception:
        return None


def bench_ba(a, local_rank, rank, world, cores, barrier, hbm):
    """Final-BA leg (BASELINE configs[3]): LM iterations per second of b2_ba_solve and the HBM
    roofline of the Jacobian+Schur kernels; CPU baseline = the reference's vendored PBA."""
    from dagsfm_b200 import BundleAdjuster, BundleAdjustmentOptions
    from dagsfm_b200.ba_scene import copy_problem, make_ba_problem, reprojection_rms
    n_img, n_pts, track = (int(x) for x in a.ba.split(","))
    prob0 = make_ba_problem(n_img=n_img, n_pts=n_pts, track_len=track, seed=1)
    n_obs = len(prob0["obs_img"])
    n_obs_total = n_obs
    opt = BundleAdjustmentOptions.default()
    opt.linear_solver_type = {"auto": 0, "exact": 1, "iterative": 2}[a.ba_solver]
    ba = BundleAdjuster(opt, device=local_rank)
    full0 = prob0
    if world > 1:   # points sharded over the ranks, one NCCL all-reduce of (S, rhs, g_c, diag) per LM iteration
        import torch
        from dagsfm_b200.parallel import make_torch_allreduce, shard_ba_problem
        prob0, _ids = shard_ba_problem(full0, rank, world)
        if os.environ.get("B2_BENCH_BA_HOOK") == "torch":     # A/B: the caller-supplied hook (host callback per all-reduce)
            ba.set_allreduce(make_torch_allreduce(torch.device("cuda", local_rank)))
        else:                                                  # the library's own communicator: ncclAllReduce on the solver stream
            ba.init_nccl_from_torch()
    prob = copy_problem(prob0)
    ba.Solve(prob)                                    # warm-up (cuSOLVER workspace, clocks)
    prob = copy_problem(prob0)
    barrier()
    t0 = time.perf_counter()
    s = ba.Solve(prob)
    barrier()
    wall = time.perf_counter() - t0
    iters = s.num_iterations + (1 if s.termination_type == 0 else 0)   # the converged check costs one build
    D = 8 * n_img - 7 - 0   # pose 6 + f,k per image, minus the 7 gauge parameters
    # algorithmic bytes per LM iteration (SURVEY 8d): 24 N_obs + 28 N_pts + 88 N_cam reads,
    # 72 N_pts + 64 N_cam + 8 * (upper triangle of the dense reduced system) writes
    alg_bytes = 24 * n_obs + 28 * n_pts + 88 * n_img + 72 * n_pts + 64 * n_img + 8 * (D * (D + 1) // 2)
    schur_ms = 1e3 * s.schur_kernel_seconds / max(iters, 1)       # every pass of the LM loop builds the system once
    achieved = alg_bytes / (schur_ms * 1e-3) / 1e9
    out = {"workload": f"{n_img} cams / {n_pts} pts / {n_obs} obs, track {track}, SIMPLE_RADIAL, final-BA options",
           "lm_iter_per_s": s.num_iterations / s.solve_seconds, "lm_iterations": s.num_iterations,
           "successful": s.num_successful_steps, "unsuccessful": s.num_unsuccessful_steps,
           "termination": s.termination_type, "solve_s": s.solve_seconds, "e2e_s": wall,
           "rms_px_initial": reprojection_rms(prob0), "rms_px_final": reprojection_rms(prob),
           "mean_reproj_error_px_final": _mean_reproj(prob),
           "rms_note": "this rank's point shard" if world > 1 else "all observations",
           "sharding": "single GPU" if world == 1 else
                       (f"points over {world} ranks, 1 ncclAllReduce (library-owned communicator, solver stream) of D doubles per inner CG iteration "
                        "(+ rhs / preconditioner blocks once per LM iteration)" if s.linear_solver_type_used == 2 else
                        f"points over {world} ranks, 1 ncclAllReduce (library-owned communicator, solver stream) of the packed reduced camera system per LM iteration"),
           "ceres_style_px": float(np.sqrt(s.final_cost / (2 * n_obs))),
           "roofline": {"bound": "hbm", "kernel": "camera_terms_kernel + schur_points_kernel + schur_window_kernel (Jacobian + Schur complement)", "achieved": achieved,
                        "peak": hbm[0] * world, "unit": "GB/s", "frac": achieved / (hbm[0] * world),
                        "peak_source": hbm[1] + (f" x {world} GPUs (whole-job bytes against the aggregate)" if world > 1 else ""),
                        "algorithmic_bytes_per_iteration": alg_bytes, "avg_ms_per_iteration": schur_ms,
                        "share_of_solve": s.schur_kernel_seconds / s.solve_seconds, "traffic": None,
                        "note": "algorithmic bytes count the full upper triangle of S as SURVEY 8d does; see DESIGN.md section 3"}}
    out["linear_solver"] = ("ITERATIVE_SCHUR + SCHUR_JACOBI" if s.linear_solver_type_used == 2 else
                            "exact Schur step: fused kernels, packed tiles, own tiled Cholesky" if s.exact_path_used == 2 else
                            "exact Schur step: staged blocks, dense S, cuSOLVER (fallback path)")
    out["linear_solve_ms_per_iteration"] = 1e3 * s.linear_solve_seconds / max(iters, 1)
    out["reduced_system_mb"] = s.reduced_system_bytes / 1e6
    out["ms_per_lm_iteration"] = 1e3 * s.solve_seconds / max(iters, 1)
    if s.linear_solver_type_used == 2:
        # matrix-free Schur product: both passes stream the 224 B Jacobian block of every observation once per CG
        # iteration (+ 12 B of indices), z_p is written and read once (DESIGN.md section 3)
        cg = max(int(s.num_linear_solver_iterations), 1)
        alg_cg = (2 * 224 + 12) * n_obs + 2 * 24 * n_pts
        lin_ms = 1e3 * s.schur_kernel_seconds / cg
        out["cg_iterations"] = int(s.num_linear_solver_iterations)
        out["roofline"] = {"bound": "hbm", "kernel": "matvec_point_kernel + image_pass_kernel<0> (per CG iteration; includes the "
                           "preconditioner set-up and the host-side reductions of the inner solve)",
                           "achieved": alg_cg / (lin_ms * 1e-3) / 1e9, "peak": hbm[0] * world, "unit": "GB/s",
                           "frac": alg_cg / (lin_ms * 1e-3) / 1e9 / (hbm[0] * world),
                           "peak_source": hbm[1] + (f" x {world} GPUs (whole-job bytes against the aggregate)" if world > 1 else ""),
                           "algorithmic_bytes_per_cg_iteration": alg_cg, "avg_ms_per_cg_iteration": lin_ms,
                           "share_of_solve": s.schur_kernel_seconds / s.solve_seconds, "traffic": None}
    if (n_img, n_pts, track) == (500, 100000, 10) and world == 1 and s.linear_solver_type_used != 2 and s.exact_path_used == 2:
        # committed ncu capture of one iteration at exactly this workload (profiles/r2_ba_fused_ncu_full.txt): camera_terms 31.5 MB,
        # schur_points 49.8 + 217.5 MB (it writes the 240 B / observation Z that schur_window reads back), schur_window 254.8 + 3.6 MB
        out["roofline"]["traffic"] = 557.2e6
        out["roofline"]["traffic_source"] = "profiles/r2_ba_fused_ncu_full.txt (dram bytes read + written per LM iteration, three kernels)"
    if rank == 0 and not a.no_cpu:
        from oracle import pyoracle as orc
        if orc.pba_ref_available():
            pc = copy_problem(full0)
            big = n_obs_total > 4_000_000          # bounded sample: a C5-size problem gets two LM iterations of the CPU reference
            r = orc.pba_ref_solve(pc, n_threads=cores, max_iter=2 if big else 50)
            out["cpu_baseline"] = {"value": r["lm_iterations"] / r["seconds"], "unit": "LM iter/s", "cores": cores,
                                   "kind": "reference", "sample": f"vendored PBA CPU double, {r['lm_iterations']} LM iterations, {r['seconds']:.1f} s"
                                                                   + (" (bounded: 2 iterations)" if big else ""),
                                   "final_mse_px2": float(r["final_mse"]),
                                   "gpu_final_mse_px2": float(2 * s.final_cost / n_obs)}
    ba.close()
    return out


FP64_PEAK_FALLBACK = 36.6   # TFLOP/s, DFMA micro-benchmark on this pool's B200 (profiles/r2_fp64_peak.json)


def peaks_fp64():
    try:
        d = json.loads((ROOT / "profiles" / "r2_fp64_peak.json").read_text())
        return float(d["fp64_tflops"]), "profiles/r2_fp64_peak.json (b2_peak_fp64 DFMA micro-benchmark on a pool B200; MEASURED_PEAKS.json has no FP64 entry)"
    except Exception:
        return FP64_PEAK_FALLBACK, "fallback: 36.6 TFLOP/s measured on a pool B200 in round 2"


def pipeline_cpu_reference(coll_desc_host, keypoints, cam_params, prior, pairs, seeds, n_sample, threads):
    """The reference's CPU path for the pipeline on a uniform sample of the step's pairs: MatchSiftFeaturesCPU
    (oracle port of sift.cc:76-198,810-822) then TwoViewGeometry::Estimate (oracle port of two_view_geometry.cc:292-489),
    `threads` workers each on one pair at a time (matching.cc:640-660).  -> (pairs/s, seconds, sample indices,
    oracle results, oracle match counts)."""
    import ctypes as C
    from concurrent.futures import ThreadPoolExecutor
    from oracle import pyoracle as orc
    rng = np.random.default_rng(0)
    idx = np.sort(rng.choice(len(pairs), size=min(n_sample, len(pairs)), replace=False))
    sample = np.ascontiguousarray(pairs[idx])
    ns = len(sample)
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads) as ex:      # ctypes releases the GIL inside the oracle
        mts = list(ex.map(lambda ab: orc.match_sift(coll_desc_host[ab[0]], coll_desc_host[ab[1]]), sample.tolist()))
    t_match = time.perf_counter() - t0
    off = np.concatenate([[0], np.cumsum([len(m) for m in mts])]).astype(np.int64)
    mt = np.ascontiguousarray(np.concatenate(mts) if off[-1] else np.zeros((0, 2), np.uint32), dtype=np.uint32)
    n_img = len(keypoints)
    ocams = (orc.OrcCamera * n_img)(*[orc.make_camera(params=cam_params, prior=bool(p)) for p in prior])
    kk = [np.ascontiguousarray(k, np.float64) for k in keypoints]
    ptrs = (C.c_void_p * n_img)(*[k.ctypes.data for k in kk])
    oo = orc.tv_default_options()
    ores = (orc.OrcTvResult * ns)()
    oinl = np.zeros((max(int(off[-1]), 1), 2), np.uint32)
    sd = np.ascontiguousarray(seeds[idx], np.uint32)
    with orc.solver_stack(1):   # the oracle in the kernel's operation order: identity with the GPU, not an agreement rate
        t_verify = orc._tv().orc_two_view_pairs_mt2(C.cast(ocams, C.c_void_p), C.cast(ptrs, C.c_void_p), sample.ctypes.data, ns,
                                                    off.ctypes.data, mt.ctypes.data, C.byref(oo), sd.ctypes.data, threads,
                                                    C.cast(ores, C.c_void_p), oinl.ctypes.data)
    secs = t_match + t_verify
    return ns / secs, secs, idx, ores, np.diff(off), (t_match, t_verify)


def bench_pipeline(a, dev, local_rank, rank, world, cores, barrier, dist):
    """C3: match -> verify of one candidate list, sharded over the ranks; see the module docstring."""
    import torch
    from dagsfm_b200 import SiftMatchingOptions, TwoViewOptions, lib
    from dagsfm_b200.pipeline import SiftFeatureMatcher, cameras_of
    from dagsfm_b200.synthetic import candidate_pairs, make_image_collection
    coll = make_image_collection(a.seq_images, a.seq_kp, seed=1234, device=dev, overlap_images=a.seq_cand)
    pairs_all = candidate_pairs(a.seq_images, a.seq_cand)
    n_all = len(pairs_all)
    seeds_all = (np.arange(n_all, dtype=np.uint64) * 2654435761 % (2 ** 32)).astype(np.uint32)
    # ONE list, dealt to the ranks in blocks of 4 096 consecutive (locality-ordered) pairs, block b to rank b mod N: every
    # rank sees every part of the sequence, so stretches that verify fast (planar scene parts) or slow spread evenly --
    # the static counterpart of the reference's shared matcher queue (feature/matching.cc:619-638)
    blk = 4096
    owner = (np.arange(n_all) // blk) % world
    idx_of = [np.nonzero(owner == r)[0] for r in range(world)]
    pairs, seeds = pairs_all[idx_of[rank]], seeds_all[idx_of[rank]]
    cams = cameras_of(coll)
    fm = SiftFeatureMatcher(SiftMatchingOptions(), TwoViewOptions.default(), local_rank, chunk_pairs=a.chunk_pairs)
    fm.setup_device_descriptors(coll["desc"].data_ptr(), a.seq_images, a.seq_kp, coll["keypoints"], cams)
    from dagsfm_b200.verification import RESULT_DTYPE
    gathered = None

    def gather(res):
        """rank 0 receives every shard's results (the reference's single output queue / database writer)."""
        nonlocal gathered
        if world == 1:
            gathered = res.copy()        # the matcher's result array is a view of its pinned buffer, rewritten by the next call
            return
        t = torch.from_numpy(res.view(np.uint8).reshape(-1)).to(dev)
        sizes = [len(idx_of[r]) * RESULT_DTYPE.itemsize for r in range(world)]
        pad = torch.zeros(max(sizes), dtype=torch.uint8, device=dev)
        pad[:t.numel()] = t
        out = [torch.empty(max(sizes), dtype=torch.uint8, device=dev) for _ in range(world)] if rank == 0 else None
        dist.gather(pad, out, dst=0)
        if rank == 0:
            gathered = np.empty(n_all, RESULT_DTYPE)
            for r, (o, sz) in enumerate(zip(out, sizes)):
                gathered[idx_of[r]] = o[:sz].cpu().numpy().view(RESULT_DTYPE)

    def step():
        res, _, _, _ = fm.run_device(pairs, seeds, keep_lists=False)
        gather(res)
        return res

    for _ in range(a.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = lib().b2_kernel_launch_count()
    t_match = t_verify = 0.0
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wall0 = time.perf_counter()
    ev0.record()
    for _ in range(a.steps):
        res = step()
        t_match += fm.match_seconds
        t_verify += fm.verify_seconds
    ev1.record()
    barrier()
    wall = time.perf_counter() - wall0
    last_step = gathered
    launches = lib().b2_kernel_launch_count() - launches0
    clocks = sampler.stop()
    if world > 1:
        t = torch.tensor([wall, t_match, t_verify], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        wall, t_match, t_verify = t.tolist()
    out = {"n_pairs": n_all, "wall_s": wall, "match_kernel_s": t_match, "verify_kernel_s": t_verify,
           "launches": int(launches), "clocks": clocks, "value": n_all * a.steps / wall}
    # ------------------------------------------------------------------ e2e: host buffers in, results + lists out
    if not a.no_e2e:
        host = torch.empty(coll["desc"].shape, dtype=torch.uint8, pin_memory=True)
        host.copy_(coll["desc"])
        hd = host.numpy()
        hdescs = [hd[i] for i in range(a.seq_images)]
        kps = list(coll["keypoints"])
        e_steps = a.steps
        d2h = 0
        t_setup = t_run = 0.0

        def e2e_step():
            nonlocal d2h, t_setup, t_run
            t0 = time.perf_counter()
            fm.Setup(hdescs, kps, cams)                                   # H2D: descriptors + keypoints + cameras
            t1 = time.perf_counter()
            r2, off2, mt2, inl2 = fm.run_device(pairs, seeds, keep_lists=True)   # H2D pairs + seeds; D2H results + lists
            gather(r2)
            t_setup += t1 - t0
            t_run += time.perf_counter() - t1
            d2h = r2.nbytes + off2.nbytes + mt2.nbytes + inl2.nbytes

        e2e_step()          # one untimed pass: the pinned output buffers of the chain are allocated once, as a caller's would be
        t_setup = t_run = 0.0
        barrier()
        w0 = time.perf_counter()
        for _ in range(e_steps):
            e2e_step()
        barrier()
        w = time.perf_counter() - w0
        if world > 1:
            t = torch.tensor([w], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            w = t.item()
        out["e2e"] = {"value": n_all * e_steps / w, "unit": UNIT,
                      "h2d_bytes_per_step": int(hd.nbytes + coll["keypoints"].nbytes + pairs.nbytes + seeds.nbytes),
                      "d2h_bytes_per_step": int(d2h), "steps": e_steps, "warmup": 1,
                      "setup_s_per_step": t_setup / e_steps, "chain_s_per_step": t_run / e_steps,
                      "api": "SiftFeatureMatcher.Setup (b2_match_set_images + b2_verify_set_images, host buffers) + "
                             "b2_match_pairs_device -> b2_verify_pairs_device per chunk of pairs (--chunk-pairs), results / match lists / inlier lists to the host",
                      "bytes_note": "per rank" if world > 1 else "whole job"}
        fm.setup_device_descriptors(coll["desc"].data_ptr(), a.seq_images, a.seq_kp, coll["keypoints"], cams)
    if rank == 0:
        g = gathered
        m = np.maximum(g["E_num_trials"].astype(np.float64) + g["F_num_trials"], 0)
        out["results"] = {"config_histogram": {int(k): int(c) for k, c in zip(*np.unique(g["config"], return_counts=True))},
                          "mean_inliers_of_verified": float(g["n_inliers"][g["config"] > 1].mean()) if (g["config"] > 1).any() else 0.0,
                          "trials_per_pair": {k: float(g[k + "_num_trials"].mean()) for k in ("E", "F", "H")}}
        out["_gathered"], out["_last_step"] = g, last_step
    out["_coll"], out["_pairs"], out["_seeds"], out["_fm"] = coll, pairs_all, seeds_all, fm
    return out


def bench_retrieval_sharded(a, coll, local_rank, rank, world, barrier, dist, pairs_all):
    """The retrieval stage on N GPUs: every rank searches the visual words of its images, ONE all-gather of the word ids
    (NCCL), every rank builds the same inverted index and queries its own images, rank 0 gathers the candidate pairs."""
    import torch
    from dagsfm_b200.retrieval import VocabSimilarityGraph
    from dagsfm_b200.synthetic import make_vocabulary_device
    n_img, n_kp = a.seq_images, a.seq_kp
    box = [make_vocabulary_device(coll["desc"], a.retrieval_words, n_train=min(1 << 20, n_img * n_kp), seed=7) if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    g = VocabSimilarityGraph(box[0], num_images=2 * a.seq_cand, num_nearest_neighbors=5, device=local_rank)
    walls = []
    pairs = None
    for s in range(a.warmup + a.steps):
        barrier()
        t0 = time.perf_counter()
        pairs, _sc = g.RunSharded(coll["desc"], rank, world, dist)
        barrier()
        walls.append(time.perf_counter() - t0)
    w = float(np.mean(walls[a.warmup:]))
    t = torch.tensor([g.timing.get("word_search_s", 0.0), g.timing.get("index_build_s", 0.0), g.timing.get("query_s", 0.0)],
                     dtype=torch.float64, device=coll["desc"].device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank != 0:
        return None
    got = set(map(tuple, pairs.tolist()))
    near = pairs_all[(pairs_all[:, 1].astype(np.int64) - pairs_all[:, 0]) <= max(a.seq_cand // 2, 1)]
    return {"workload": f"{n_img} images x {n_kp} descriptors, {a.retrieval_words} visual words, num_neighbors 5, max_num_images {2 * a.seq_cand}",
            "images_per_s": n_img / w, "wall_s_per_step": w, "word_search_s": t[0].item(), "index_build_s": t[1].item(), "query_s": t[2].item(),
            "timing_note": "kernel times = max over ranks of the last step; wall = the whole stage incl. the all-gather and the gather of the pairs",
            "candidate_pairs": len(pairs),
            "recall_of_overlapping_pairs": float(np.mean([tuple(p) in got for p in near.tolist()])) if len(near) else None,
            "sharding": f"word search and queries of {n_img} images over {world} ranks (contiguous image ranges), 1 all-gather of the word ids "
                        f"({n_img * n_kp * 5 * 4 / 1e6:.0f} MB) per step, inverted index replicated, candidate pairs gathered on rank 0"}


def bench_retrieval(a, coll, local_rank, cores, pairs_all):
    """SURVEY 8f rank 3 / the input stage of C3: VocabSimilarityGraph::Run (similarity_graph.cpp:101-200) over the C3
    collection resident in HBM -- exact nearest visual words of every descriptor, inverted index, query of every image,
    top `seq_cand` images each.  One step = the whole stage (index + query).  Rank 0 only (the stage is not sharded)."""
    import torch
    from dagsfm_b200.retrieval import VisualIndex
    from dagsfm_b200.synthetic import make_vocabulary_device
    n_img, n_kp, K = a.seq_images, a.seq_kp, 5
    vocab = make_vocabulary_device(coll["desc"], a.retrieval_words, n_train=min(1 << 20, n_img * n_kp), seed=7)
    vi = VisualIndex(local_rank)
    n_ret = 2 * a.seq_cand      # VocabSimilaritySearchOptions::num_images = 100 (similarity_graph.h:44): the seq_cand successors + predecessors
    out = {"workload": f"{n_img} images x {n_kp} descriptors, {a.retrieval_words} visual words, num_neighbors {K}, "
                       f"max_num_images {n_ret} (VocabSimilaritySearchOptions defaults: 100 / 5)"}
    try:
        vi.set_vocabulary(vocab)
        steps = []
        for s in range(a.warmup + a.steps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            vi.index_images_device(coll["desc"].data_ptr(), n_img, n_kp, K)
            ids, sc, cnt = vi.query_all(n_ret)
            w = time.perf_counter() - t0
            if s >= a.warmup:
                steps.append((w, vi.last_timing()))
        w = float(np.mean([x[0] for x in steps]))
        tm = {k: float(np.mean([x[1][k] for x in steps])) for k in steps[0][1]}
        ops = 2.0 * 128 * n_img * n_kp * a.retrieval_words
        q = np.repeat(np.arange(n_img), ids.shape[1]).reshape(ids.shape)
        valid = (np.arange(ids.shape[1])[None, :] < cnt[:, None]) & (q < ids)
        got = set(map(tuple, np.stack([q[valid], ids[valid]], 1).tolist()))
        near = pairs_all[(pairs_all[:, 1].astype(np.int64) - pairs_all[:, 0]) <= max(a.seq_cand // 2, 1)]
        out.update({"images_per_s": n_img / w, "wall_s_per_step": w, **{k: v for k, v in tm.items()},
                    "candidate_pairs": int(valid.sum()),
                    "recall_of_overlapping_pairs": float(np.mean([tuple(p) in got for p in near.tolist()])) if len(near) else None,
                    "recall_note": f"share of the sequence's pairs up to {max(a.seq_cand // 2, 1)} images apart (>= half the scene points in common) found among the candidates",
                    "recall_of_the_pipeline_list": float(np.mean([tuple(p) in got for p in pairs_all[::max(len(pairs_all) // 20000, 1)].tolist()])),
                    "roofline": {"bound": "int8 (dp4a / tensor)", "kernel": "word_knn_kernel<5> (exact nearest words)", "unit": "TOP/s",
                                 "achieved": ops / tm["word_search_s"] / 1e12,
                                 "algorithmic_ops": "2 x 128 per descriptor x word", "share_of_step": tm["word_search_s"] / w}})
        # parity spot check + CPU baseline of the dominant part on a bounded sample (exact word search, OpenMP)
        if not a.no_cpu:
            from oracle import pyoracle as orc
            o = orc.RetrievalOracle(vocab.words, vocab.proj, vocab.thresholds, vocab.has_embedding)
            rng = np.random.default_rng(1)
            n_s = min(12288 * cores, n_img * n_kp)   # ~10 s of exact search on the host cores
            pick = np.sort(rng.choice(n_img * n_kp, n_s, replace=False))
            sample = coll["desc"].reshape(-1, 128)[torch.from_numpy(pick).to(coll["desc"].device)].cpu().numpy()
            try:      # torchrun exports OMP_NUM_THREADS=1; the oracle's word search is an OpenMP loop and gets all host cores here
                import ctypes
                ctypes.CDLL("libgomp.so.1").omp_set_num_threads(int(cores))
            except OSError:
                pass
            t0 = time.perf_counter()
            exp = o.word_ids(sample, K)
            t = time.perf_counter() - t0
            gotw = vi.debug_word_ids()[pick]
            out["cpu_baseline"] = {"value": n_s / t / n_kp, "unit": "images/s (word search only)", "cores": cores, "kind": "port",
                                   "sample": f"exact 5 nearest words of {n_s} sampled descriptors, {t:.1f} s (the reference's FLANN search is approximate and cheaper)",
                                   "identical_to_gpu": f"{int((gotw == exp).all(1).sum())}/{n_s}"}
    finally:
        vi.close()
    return out


def bench_match(a, dev, local_rank, rank, world, barrier, dist):
    """C2 leg (BASELINE configs[1]): exhaustive descriptor matching of 1000 x 4096 images, descriptors resident in HBM;
    every rank matches its own replica of the pair list (extra leg, not the headline)."""
    import torch
    from dagsfm_b200 import SiftMatchGPU, SiftMatchingOptions
    desc = make_descriptors_torch(a.images, a.desc, 1234 + rank, dev)
    pairs = all_pairs(a.images, a.pairs)
    n_pairs = len(pairs)
    opt = SiftMatchingOptions()
    m = SiftMatchGPU(local_rank)
    torch.cuda.synchronize()
    m.set_images_device(desc.data_ptr(), np.arange(a.images, dtype=np.int64) * a.desc, np.full(a.images, a.desc, dtype=np.int32))
    pairs_dev = torch.from_numpy(pairs.astype(np.int32)).to(dev)
    cap = max(64 << 20, int(n_pairs) * 64)
    off_dev = torch.empty(n_pairs + 1, dtype=torch.int64, device=dev)
    mat_dev = torch.empty((cap, 2), dtype=torch.int32, device=dev)
    steps, warm = a.steps, a.warmup
    for _ in range(warm):
        m.match_pairs_device(n_pairs, pairs_dev.data_ptr(), opt, off_dev.data_ptr(), mat_dev.data_ptr(), cap)
    barrier()
    t_dev = t_tc = 0.0
    n_tc = 0
    for _ in range(steps):
        total = m.match_pairs_device(n_pairs, pairs_dev.data_ptr(), opt, off_dev.data_ptr(), mat_dev.data_ptr(), cap)
        tm = m.last_timing()
        t_dev += tm["all_kernels_s"]
        t_tc += tm["tc_kernel_s"]
        n_tc += tm["tc_launches"]
    barrier()
    if world > 1:
        t = torch.tensor([t_dev], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_dev = t.item()
    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained") or 1400.0
    ops_per_pair = 2.0 * a.desc * a.desc * 128
    achieved = ops_per_pair * n_pairs * steps / t_tc / 1e12
    i8 = None
    try:
        i8 = json.loads((ROOT / "profiles" / "r2_fp64_peak.json").read_text()).get("i8_tops_library_gemm")
    except Exception:
        pass
    out = {"workload": f"C2: {a.images} images x {a.desc} desc, {n_pairs} pairs per step ({'exhaustive' if n_pairs == a.images * (a.images - 1) // 2 else 'prefix of the exhaustive list'}), replicated per rank",
           "pairs_per_s": world * n_pairs * steps / t_dev, "ms_per_step": 1e3 * t_dev / steps, "matches_per_step": int(total),
           "roofline": {"bound": "tensor", "kernel": "match_top2_ts_kernel (tcgen05 kind::i8, query operand in TMEM)",
                        # the denominator is an i8 rate measured on this pool's B200s: the cuBLASLt u8/s8 GEMM (profiles/r2_fp64_peak.json);
                        # MEASURED_PEAKS.json's bf16 figure is kept beside it.  `achieved` counts a pair ONCE (algorithmic); the kernel
                        # contracts it twice (one pass per direction), which `executed_frac` shows.
                        "achieved": achieved, "unit": "TOP/s",
                        "peak": i8 if i8 else peak_tf,
                        "frac": achieved / (i8 if i8 else peak_tf),
                        "executed_frac": (2 * achieved / i8) if i8 else None,
                        "peak_source": ("profiles/r2_fp64_peak.json i8_tops_library_gemm (cuBLASLt i8 GEMM on a pool B200)" if i8 else
                                        "MEASURED_PEAKS.json bf16_tflops_sustained (no i8 measurement found)"),
                        "frac_of_bf16_sustained": achieved / peak_tf,
                        "bf16_peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback 1.4 PFLOP/s",
                        "algorithmic_ops_per_pair": ops_per_pair, "avg_launch_ms": 1e3 * t_tc / max(n_tc, 1), "launches": n_tc,
                        "share_of_step": t_tc / t_dev, "traffic": 4.534e9 if (a.desc == 4096 and n_tc and abs(n_pairs * steps / n_tc - 8192) < 64) else None}}
    m.close()
    return out


def main():
    a = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cores = effective_cores()
    if a.c1:
        a.seq_images, a.seq_kp, a.seq_cand = 100, 2048, 99      # every successor = the exhaustive pair list
        a.cpu_sample, a.pairs, a.ba, a.ba_c5 = 4950, -1, "", ""
        a.retrieval_words = min(a.retrieval_words, 4096)
    if a.cpu_sample <= 0:
        a.cpu_sample = 24 * cores      # ~10-20 s of host work at ~2 pairs per core-second
    n_cand = a.seq_images * a.seq_cand - a.seq_cand * (a.seq_cand + 1) // 2
    workload = (f"{'C1 (exhaustive pairs)' if a.c1 else 'C3'}: {a.seq_images} images x {a.seq_kp} keypoints, {a.seq_cand} candidate pairs per image ({n_cand} pairs), "
                f"descriptor match + ratio test + cross check -> E/F/H LO-RANSAC verification, chained on the device")
    cfg = {"workload": workload, "n_images": a.seq_images, "keypoints_per_image": a.seq_kp, "candidates_per_image": a.seq_cand,
           "options": "match: max_ratio 0.8, max_distance 0.7, cross_check 1; verify: reference defaults (max_error 4 px, confidence 0.999, "
                      "max_num_trials 10000, min_inlier_ratio 0.25, min_num_inliers 15)",
           "l2": (lambda mib: f"descriptor pool {mib:.0f} MiB " + ("> 126 MB L2 (inputs larger than L2)" if mib > 126
                                                                     else "<= 126 MB L2 (NOT a valid timing configuration)"))(
               a.seq_images * a.seq_kp * 128 / 2**20),
           "sharding": "one candidate list dealt to the ranks in blocks of 4 096 consecutive pairs (block b -> rank b mod N), results gathered on rank 0 in list order (no data-path collective)"}

    import torch

    # ------------------------------------------------------------ reference arm
    if a.impl == "reference":
        if rank != 0:
            return
        from dagsfm_b200.synthetic import candidate_pairs, make_image_collection
        dev = "cuda" if torch.cuda.is_available() else "cpu"
        coll = make_image_collection(a.seq_images, a.seq_kp, seed=1234, device=dev, overlap_images=a.seq_cand)
        hd = coll["desc"].cpu().numpy()
        pairs = candidate_pairs(a.seq_images, a.seq_cand)
        seeds = (np.arange(len(pairs), dtype=np.uint64) * 2654435761 % (2 ** 32)).astype(np.uint32)
        from oracle import pyoracle as orc
        orc.lib()
        per = []
        for s in range(a.warmup + a.steps):
            v, secs, *_ = pipeline_cpu_reference(hd, coll["keypoints"], coll["cam_params"], coll["prior"], pairs, seeds,
                                                 a.cpu_sample, cores)
            if s >= a.warmup:
                per.append((v, secs))
        v = float(np.mean([p[0] for p in per]))
        ms = float(np.mean([p[1] for p in per])) * 1e3
        sample = f"{a.cpu_sample} uniformly sampled candidate pairs of the step per timed step, match + verify, {cores} threads"
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64 (verification) / u8 x u8 -> s32 (matching)", "data": "synthetic",
            "config": cfg,
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return

    # ----------------------------------------------------------------- our arm
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        # NCCL prints its version banner on stdout at the first collective; keep stdout for the
        # one JSON line by routing fd 1 to stderr until the communicator is up
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    pl = bench_pipeline(a, dev, local_rank, rank, world, cores, barrier, dist)
    fm = pl.pop("_fm")
    coll, pairs_all, seeds_all = pl.pop("_coll"), pl.pop("_pairs"), pl.pop("_seeds")
    gathered = pl.pop("_gathered", None)
    last_step = pl.pop("_last_step", None)
    if rank == 0 and a.dump_outputs:
        dump_outputs(a.dump_outputs, last_step, pairs_all)

    # ------------------------------------------------------------------ CPU baseline + parity spot check (rank 0)
    cpu = None
    if rank == 0 and not a.no_cpu:
        hd = coll["desc"].cpu().numpy()
        v, secs, idx, ores, ocounts, (tm, tv) = pipeline_cpu_reference(hd, coll["keypoints"], coll["cam_params"], coll["prior"],
                                                                      pairs_all, seeds_all, a.cpu_sample, cores)
        g = gathered[idx]
        same = sum(int(ores[i].config == g["config"][i] and ores[i].n_inliers == g["n_inliers"][i] and
                       ores[i].E_trials == g["E_num_trials"][i] and ores[i].F_trials == g["F_num_trials"][i] and
                       ores[i].H_trials == g["H_num_trials"][i] and
                       all(np.array_equal(np.array(getattr(ores[i], m)[:]).view(np.uint64), g[m][i].view(np.uint64)) for m in "EFH"))
                   for i in range(len(idx)))
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{len(idx)} uniformly sampled candidate pairs of the step, {secs:.1f} s ({tm:.1f} s matching + {tv:.1f} s verification), "
                         "oracle port of MatchSiftFeaturesCPU + TwoViewGeometry::Estimate",
               "identical_to_gpu": f"{same}/{len(idx)}",
               "identical_means": "configuration, inlier and trial counts, E / F / H bit for bit, on matches the oracle computed itself"}
    fm.close()
    retrieval = None
    if a.retrieval_words > 0 and world > 1:
        retrieval = bench_retrieval_sharded(a, coll, local_rank, rank, world, barrier, dist, pairs_all)   # collective: every rank
    elif rank == 0 and a.retrieval_words > 0:
        try:
            retrieval = bench_retrieval(a, coll, local_rank, cores, pairs_all)
        except Exception as e:   # an extra leg must not take the headline line down
            retrieval = {"error": repr(e)}
    del coll
    torch.cuda.empty_cache()

    # ------------------------------------------------------- extra legs
    match = bench_match(a, dev, local_rank, rank, world, barrier, dist) if a.pairs >= 0 else None
    verify = bench_verify(a, local_rank, rank, world, cores, barrier) if a.verify_pairs > 0 else None
    guided = None
    if getattr(a, "guided_pairs", 0) > 0:
        try:
            guided = bench_guided(a, local_rank, rank, world, cores, barrier)
        except Exception as e:
            guided = {"error": repr(e)}
    ba = bench_ba(a, local_rank, rank, world, cores, barrier, peaks_hbm()) if a.ba else None
    ba_c5 = None
    if a.ba_c5:
        import copy
        a5 = copy.copy(a)
        a5.ba, a5.ba_solver = a.ba_c5, "auto"
        try:
            ba_c5 = bench_ba(a5, local_rank, rank, world, cores, barrier, peaks_hbm())
        except Exception as e:   # an extra leg must not take the headline line down
            ba_c5 = {"error": repr(e)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # --------------------------------------------------------------- roofline of the dominant kernel of the step
    # verify_pairs_kernel: SURVEY 8(d) unit = one hypothesis evaluated against one match (33 FP64 flop Sampson for E / F,
    # 25 for H); lower bound from the trial counts the kernel reports (>= 1 hypothesis per trial, LO and tie passes not
    # counted), divided by the kernel's device time (CUDA events on its stream) -- FP64 vector work, not HBM or tensor.
    peak64, peak64_src = peaks_fp64()
    g = gathered
    mcount = None
    roofline = {"bound": "fp64", "kernel": "verify_stage_kernel<E|F|H|decision> (one warp per pair, 32 RANSAC trials per batch; the H stage is ~65 % of it)", "unit": "TFLOP/s",
                "peak": peak64, "peak_source": peak64_src,
                "share_of_step": pl["verify_kernel_s"] / max(pl["verify_kernel_s"] + pl["match_kernel_s"], 1e-12),
                "avg_launch_ms": 1e3 * pl["verify_kernel_s"] / max(a.steps * ((pl["n_pairs"] // world + a.chunk_pairs - 1) // a.chunk_pairs), 1),
                "launch_note": "one launch = the four stage kernels (E, F, H, decision) of one chunk of pairs"}
    # dram__bytes_read + write of the three RANSAC stage kernels in the committed capture (profiles/r2_verify_final_ncu_full.txt:
    # 3.96 + 2.94 + 4.49 GB for a 13 725-pair launch group at 2 048 keypoints per image = 0.83 MB per pair, mostly the per-warp
    # scratch -- hypotheses, local-optimisation matrices -- spilling past L2), scaled to this run's pairs per launch
    pairs_per_launch = min(a.chunk_pairs, max(pl["n_pairs"] // world, 1))
    roofline["traffic"] = 11.39e9 / 13725 * pairs_per_launch
    roofline["traffic_source"] = "profiles/r2_verify_final_ncu_full.txt (bytes per pair of the 2 048-keypoint capture x pairs per launch)"
    try:
        off = None
        # matches per pair are not kept by the throughput run: expected count from the scene layout (shared points +
        # distractors of the overlap), exact enough for a lower bound that is itself a lower bound
        d = (pairs_all[:, 1].astype(np.int64) - pairs_all[:, 0].astype(np.int64))
        shared, stride = a.seq_kp // 2, max((a.seq_kp // 2) // a.seq_cand, 1)
        n_dis = int(a.seq_kp * 0.125)
        dstride = max(n_dis // a.seq_cand, 1)
        mexp = np.maximum(shared - d * stride, 0) + np.maximum(n_dis - d * dstride, 0)
        ef = (g["E_num_trials"].astype(np.float64) + g["F_num_trials"]) * mexp
        hh = g["H_num_trials"].astype(np.float64) * mexp
        flops = a.steps * float(33.0 * ef.sum() + 25.0 * hh.sum())
        roofline["peak"] = peak64 * world
        if world > 1:
            roofline["peak_source"] = peak64_src + f" x {world} GPUs (whole-job flops against the aggregate)"
        roofline.update({"achieved": flops / pl["verify_kernel_s"] / 1e12, "frac": flops / pl["verify_kernel_s"] / 1e12 / (peak64 * world),
                         "algorithmic_flop_per_unit": "33 (E, F Sampson) / 25 (H transfer) per hypothesis x match",
                         "units_per_step_min": float(ef.sum() + hh.sum()), "mean_matches_per_pair_expected": float(mexp.mean())})
    except Exception as e:
        roofline["error"] = repr(e)

    e2e = pl.pop("e2e", None)
    print(json.dumps({
        "metric": METRIC, "value": pl["value"], "unit": UNIT, "n_gpus": world, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * pl["wall_s"] / a.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64 (verification) / u8 x u8 -> s32 exact (matching)", "data": "synthetic",
        "config": cfg, "e2e": e2e, "gpu_launches": pl["launches"], "clocks": pl["clocks"],
        "roofline": roofline, "cpu_baseline": cpu,
        "pipeline": {"pairs_per_step": pl["n_pairs"], "match_kernel_ms_per_step": 1e3 * pl["match_kernel_s"] / a.steps,
                     "verify_kernel_ms_per_step": 1e3 * pl["verify_kernel_s"] / a.steps,
                     "timing": "value = pairs / wall time of the K steps between device synchronisations (kernels, chunk "
                               "hand-over, result gather); *_kernel_ms = CUDA-event time of the two stages on their streams, max over ranks",
                     **pl.get("results", {})},
        "retrieval": retrieval, "match": match, "verify": verify, "ba": ba, "ba_c5": ba_c5, **({"guided": guided} if guided is not None else {}),
    }), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

"""Generates tests/golden/retrieval_flann_linear.npz from the reference's VENDORED FLANN (lib/FLANN, built by oracle/Makefile
into oracle/_ref/libflann_ref.so): the k nearest visual words of a descriptor set by flann::LinearIndex over flann::L2<uint8>,
i.e. the reference's own distance functor and result set in exact mode, on a vocabulary that contains duplicate words (exact
distance ties); and tests/golden/retrieval_flann_random.npz, the same search on the random cases of
tests/test_oracle_retrieval.py.  Run where the reference tree exists:
    make -C oracle ref && python tests/golden/make_retrieval_flann_golden.py"""
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

from oracle import pyoracle as orc  # noqa: E402


def linear():
    rng = np.random.default_rng(2024)
    base = rng.integers(0, 256, (40, 128)).astype(np.uint8)
    words = np.clip(base[rng.integers(0, 40, 150)].astype(np.int16) + rng.integers(-12, 13, (150, 128)), 0, 255).astype(np.uint8)
    words[7] = words[3]; words[90] = words[3]; words[41] = words[120]; words[13] = words[149]   # exact ties
    desc = np.clip(base[rng.integers(0, 40, 300)].astype(np.int16) + rng.integers(-20, 21, (300, 128)), 0, 255).astype(np.uint8)
    out = {"words": words, "desc": desc}
    for k in (1, 2, 5, 8):
        ids, dist = orc.flann_ref_knn_linear(words, desc, k)
        out[f"ids_k{k}"] = ids
        out[f"dist_k{k}"] = dist
    np.savez_compressed(ROOT / "tests" / "golden" / "retrieval_flann_linear.npz", **out)
    print("written", {k: v.shape for k, v in out.items()})


def random_cases():
    from tests.test_oracle_retrieval import flann_case_digest, flann_random_cases
    out = {}
    for i, (words, desc, k) in enumerate(flann_random_cases()):
        out[f"ids_{i}"], _ = orc.flann_ref_knn_linear(words, desc, k)
        out[f"digest_{i}"] = np.array(flann_case_digest(words, desc, k))
    np.savez_compressed(ROOT / "tests" / "golden" / "retrieval_flann_random.npz", **out)
    print("written", {k: v.shape for k, v in out.items()})


def main():
    assert orc.flann_ref_available(), "build oracle/_ref first (make -C oracle ref, needs the reference tree)"
    linear()
    random_cases()


if __name__ == "__main__":
    main()

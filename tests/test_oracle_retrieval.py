"""The retrieval oracle (oracle/retrieval_oracle.cc) against what the reference's own tests pin
(src/retrieval/visual_index_test.cc:84-112: an indexed image queried with its own descriptors ranks first with a
strictly larger score, result sizes follow max_num_images) and against a plain numpy restatement of the scoring formula
(idf weights, Hamming weights, burstiness and the two normalisations)."""
from pathlib import Path

import numpy as np

from dagsfm_b200.retrieval import make_vocabulary
from oracle import pyoracle as orc
from tests.retrieval_cases import collection, oracle_index


def test_hamming_weight_table_follows_the_functor():
    # HammingDistWeightFunctor<64, 16> (retrieval/utils.h:52-82): exp(-h^2 / 16^2) for h <= 1.5 * 16, else 0
    descs, vocab = collection(4, 64, 16)
    lut = oracle_index(descs, vocab).lut()
    h = np.arange(65, dtype=np.float32)
    assert np.allclose(lut[:25], np.exp(-h[:25] ** 2 / 256.0), rtol=1e-6) and (lut[25:] == 0).all()


def test_reference_structure_test_replayed():
    # visual_index_test.cc: 1000 random training descriptors, 100 words, two images of 50 random descriptors
    rng = np.random.default_rng(0)
    train = rng.integers(0, 256, (1000, 128)).astype(np.uint8)
    vocab = make_vocabulary(train, 100, seed=0)
    d1 = rng.integers(0, 256, (50, 128)).astype(np.uint8)
    d2 = rng.integers(0, 256, (50, 128)).astype(np.uint8)
    o = orc.RetrievalOracle(vocab.words, vocab.proj, vocab.thresholds, vocab.has_embedding)
    o.Add(1, d1); o.Add(2, d2); o.Prepare()
    ids, sc = o.Query(d1)
    assert ids.tolist() == [1, 2] and sc[0] > sc[1]
    ids, sc = o.Query(d1, max_num_images=1)
    assert ids.tolist() == [1]
    ids, sc = o.Query(d1, max_num_images=3)
    assert ids.tolist() == [1, 2] and sc[0] > sc[1]


def test_scores_equal_a_numpy_restatement_of_the_formula():
    descs, vocab = collection(8, 128, 48, seed=5)
    o = oracle_index(descs, vocab)
    cat = np.concatenate(descs)
    fimg = np.repeat(np.arange(len(descs)), [len(d) for d in descs])
    w1 = o.word_ids(cat, 1)[:, 0]
    sig = o.signatures(cat, w1)
    n_img = len(descs)
    idf = np.zeros(len(vocab.words))
    for w in np.unique(w1):
        idf[w] = np.float32(np.log(n_img / len(np.unique(fimg[w1 == w]))))
    norm = np.array([1.0 / np.sqrt((idf[w1[fimg == i]] ** 2).sum()) for i in range(n_img)])
    lut = o.lut().astype(np.float64)
    q = 3
    wid = o.word_ids(descs[q], 5)
    scores = np.zeros(n_img)
    hit = np.zeros(n_img, bool)
    for i in range(len(descs[q])):
        for w in wid[i]:
            if not vocab.has_embedding[w]:
                continue
            b = o.signatures(descs[q][i:i + 1], [w])[0]
            sel = np.where(w1 == w)[0]
            hd = np.array([bin(int(b) ^ int(s)).count("1") for s in sig[sel]])
            for im in np.unique(fimg[sel]):
                m = (fimg[sel] == im) & (hd <= 24)
                if m.any():
                    scores[im] += lut[hd[m]].sum() / np.sqrt(m.sum()) * idf[w] ** 2
                    hit[im] = True
    self_sim = (idf[wid.reshape(-1)] ** 2).sum()
    scores *= norm / np.sqrt(self_sim)
    ids, sc = o.Query(descs[q], 5, -1)
    assert set(ids.tolist()) == set(np.where(hit)[0].tolist())
    assert np.allclose(sc, scores[ids], rtol=1e-5)
    assert ids[0] == q                                  # the image itself ranks first
    assert (np.diff(sc) <= 0).all()


def test_neighbouring_images_outrank_distant_ones():
    descs, vocab = collection(14, 256, 96)
    o = oracle_index(descs, vocab)
    ids, sc = o.Query(descs[6], 5, 5)
    assert ids[0] == 6 and set(ids[1:3].tolist()) <= {4, 5, 7, 8}


# ---------------------------------------------------------------- pins against the reference's own (vendored) FLANN
def _golden():
    from pathlib import Path
    return np.load(Path(__file__).parent / "golden" / "retrieval_flann_linear.npz")


def test_exact_word_search_equals_the_references_flann_golden_vectors():
    """tests/golden/retrieval_flann_linear.npz: the reference's vendored FLANN (lib/FLANN) in exact mode -- flann::LinearIndex,
    flann::L2<uint8>, KNNResultSet -- on a vocabulary with duplicate words; generator tests/golden/make_retrieval_flann_golden.py.
    The oracle's nearest words (and through them the kernels') must be the same ids in the same order, ties included, and the
    squared distances FLANN reports must be the integers the oracle's definition gives."""
    g = _golden()
    words, desc = g["words"], g["desc"]
    o = orc.RetrievalOracle(words, np.zeros((64, 128), np.float32), np.zeros((len(words), 64), np.float32), np.ones(len(words), np.uint8))
    for k in (1, 2, 5, 8):
        ids = o.word_ids(desc, k)
        assert (ids == g[f"ids_k{k}"]).all()
        d2 = ((desc[:, None, :].astype(np.int64) - words[ids].astype(np.int64)) ** 2).sum(2)
        assert (d2 == g[f"dist_k{k}"].astype(np.int64)).all()


def flann_random_cases():
    """Random vocabularies (one word duplicated where there are more than 20) and descriptor sets: (words, desc, k) per case."""
    rng = np.random.default_rng(7)
    for n_words, n, k in ((33, 100, 5), (700, 400, 5), (1, 10, 1), (129, 64, 8)):
        words = rng.integers(0, 256, (n_words, 128)).astype(np.uint8)
        if n_words > 20:
            words[n_words // 2] = words[3]
        desc = rng.integers(0, 256, (n, 128)).astype(np.uint8)
        yield words, desc, min(k, n_words)


def flann_case_digest(words, desc, k):
    import hashlib
    return hashlib.sha256(words.tobytes() + desc.tobytes() + bytes([k])).hexdigest()


def test_exact_word_search_equals_the_vendored_flann_on_random_cases():
    """The same comparison on random cases: tests/golden/retrieval_flann_random.npz holds the nearest words the reference's
    vendored FLANN (oracle/_ref/libflann_ref.so, exact mode) returned for flann_random_cases(), with a digest of each case's
    inputs; generator tests/golden/make_retrieval_flann_golden.py."""
    g = np.load(Path(__file__).parent / "golden" / "retrieval_flann_random.npz")
    for i, (words, desc, k) in enumerate(flann_random_cases()):
        assert str(g[f"digest_{i}"]) == flann_case_digest(words, desc, k), f"case {i}: inputs differ from the stored ones"
        o = orc.RetrievalOracle(words, np.zeros((64, 128), np.float32), np.zeros((len(words), 64), np.float32), np.ones(len(words), np.uint8))
        assert (o.word_ids(desc, k) == g[f"ids_{i}"]).all()

"""
Pins the oracle (oracle/phamers_oracle.py, oracle/kmer_oracle.c) against
  (a) the committed golden vectors, which tests/golden/make_golden.py produced by running the
      UNMODIFIED reference modules, and
  (b) the original scripts themselves when PHAMERS_REF names their directory.
CPU only.
"""
import os

import numpy as np
import pytest

from oracle import phamers_oracle as po
from oracle import c_oracle
from oracle import ref_loader


def _seqs(g):
    blob, off = g["seq_bytes"].tobytes().decode("ascii"), g["seq_offsets"]
    return [blob[off[i]:off[i + 1]] for i in range(len(off) - 1)]


@pytest.fixture(scope="module")
def counting(golden_dir):
    return np.load(os.path.join(golden_dir, "counting_golden.npz"))


def test_known_answer_index_order():
    # scripts/kmer.py:90-91: "'AAAT' is at index 1 for DNA"
    assert po.count_string("AAAT", 4)[1] == 1
    assert po.count_string("ATGC", 1).tolist() == [1, 1, 1, 1]
    assert po.count_string("AATTGGCCNAa", 2).tolist() == [1, 1, 0, 0, 0, 1, 1, 0, 0, 0, 1, 1, 0, 0, 0, 1]


@pytest.mark.parametrize("k", [1, 2, 3, 4, 5, 6])
def test_python_restatements_match_golden(counting, k):
    seqs = _seqs(counting)
    want = counting["counts_k%d" % k]
    for i, s in enumerate(seqs):
        if len(s) <= 600:       # the interpreted loop only on the short cases
            got = po.count_string(s, k)
            assert got.dtype == np.int64 or got.dtype == int
            assert np.array_equal(got, want[i]), (i, s[:30])
        assert np.array_equal(po.count_string_np(s, k), want[i]), (i, s[:30])


@pytest.mark.parametrize("k", [1, 2, 3, 4, 5, 6])
def test_c_restatement_matches_golden(counting, k):
    got = c_oracle.count(counting["seq_bytes"], counting["seq_offsets"], k)
    assert np.array_equal(got, counting["counts_k%d" % k])


def test_dispatch_and_normalize(counting):
    seqs = _seqs(counting)
    one = po.count([seqs[12]], 4)
    assert one.shape == (256,) and np.array_equal(one, counting["dispatch_list1"])
    three = po.count(seqs[8:11], 4)
    assert three.shape == (3, 256) and np.array_equal(three, counting["dispatch_list3"])
    norm = po.count(seqs[13], 4, normalize=True)
    assert norm.dtype == np.float64 and np.array_equal(norm, counting["dispatch_str_norm"])
    assert po.count(12345, 4) is None
    got = po.normalize_counts(counting["counts_k4"])
    assert np.array_equal(got, counting["normalized_k4"], equal_nan=True)
    assert np.array_equal(c_oracle.normalize(counting["counts_k4"]), counting["normalized_k4"], equal_nan=True)
    assert np.isnan(got[0]).all()       # the empty sequence: 0/0 (kmer.py:219-220 has no guard)


def test_count_file_matches_golden(golden_dir, tmp_path):
    g = np.load(os.path.join(golden_dir, "fasta_golden.npz"))
    path = tmp_path / "contigs.fasta"
    with open(path, "w", newline="") as fh:
        fh.write(str(g["fasta_text"]))
    for k in (4, 5, 6):
        ids, counts = po.count_file(str(path), k, fast=True)
        assert [str(x) for x in ids] == [str(x) for x in g["ids"]]
        assert np.array_equal(counts, g["counts_k%d" % k])
    _, slow = po.count_file(str(path), 4)
    assert np.array_equal(slow, g["counts_k4"])
    _, freq = po.count_file(str(path), 4, normalize=True)
    assert np.array_equal(freq, g["freq_k4"], equal_nan=True)
    assert po.count_file(str(tmp_path / "missing.fasta"), 4) == (None, None)


def test_canonical_fold_properties():
    for k, n_canon in ((4, 136), (5, 512), (6, 2080)):
        rep, compact, n = po.canonical_map(k)
        assert n == n_canon
        # rc is an involution and the fold conserves mass
        assert all(po.revcomp_index(po.revcomp_index(j, k), k) == j for j in range(4 ** k))
        rng = np.random.default_rng(k)
        counts = rng.integers(0, 1000, size=(3, 4 ** k))
        assert np.array_equal(po.canonical_fold(counts, k).sum(axis=1), counts.sum(axis=1))
        assert po.canonical_fold(counts, k).shape == (3, n_canon)
    # a sequence and its reverse complement have the same canonical counts
    s = "ATGCGGATTTACGCGCGATATCCGATGCAAA"
    comp = {"A": "T", "T": "A", "G": "C", "C": "G"}
    rc = "".join(comp[c] for c in reversed(s))
    for k in (4, 5, 6):
        assert np.array_equal(po.canonical_fold(po.count_string(s, k), k), po.canonical_fold(po.count_string(rc, k), k))


@pytest.fixture(scope="module")
def scoring(golden_dir):
    g = np.load(os.path.join(golden_dir, "scoring_golden.npz"))
    ref = np.load(os.path.join(os.path.dirname(golden_dir), "..", "phamers_b200", "data", "reference_features.npz"))
    n_ref = int(g["n_ref"])
    pos = po.normalize_counts(ref["positive_counts"][:n_ref].astype(np.int64))
    neg = po.normalize_counts(ref["negative_counts"][:n_ref].astype(np.int64))
    return g, pos, neg


def test_scoring_restatement_matches_golden(scoring):
    g, pos, neg = scoring
    pts = po.normalize_counts(g["query_counts"])
    cents = (g["centroids_pos"], g["centroids_neg"])
    knn = po.score_points(pts, pos, neg, method="knn")
    assert np.array_equal(knn, g["scores_knn"])
    km = po.score_points(pts, pos, neg, method="kmeans", centroids=cents)
    assert np.max(np.abs(km - g["scores_kmeans"])) <= 1e-12
    combo = po.score_points(pts, pos, neg, centroids=cents)
    assert np.max(np.abs(combo - g["scores_combo"])) <= 1e-12
    assert np.all(np.abs(g["scores_combo"]) <= 1 + np.tanh(1.0) + 1e-12)   # range +-1.7616, not [-1, 1]
    # the direct-difference float64 vote agrees with scikit-learn's GEMM-trick vote on every golden query
    labels = np.append(np.ones(len(pos)), np.zeros(len(neg)))
    assert np.array_equal(po.knn_scores_exact(pts, np.vstack((pos, neg)), labels), g["scores_knn"])


def test_host_kmeans_reproduces_golden_centroids(scoring):
    # scikit-learn is the same build on the GPU box; tolerate reduction-order noise across thread counts
    g, pos, neg = scoring
    cp, cn = po.reference_centroids(pos, neg)
    assert cp.shape == (86, 256) and cn.shape == (86, 256)
    assert np.max(np.abs(cp - g["centroids_pos"])) < 1e-9
    assert np.max(np.abs(cn - g["centroids_neg"])) < 1e-9


def test_restatement_matches_live_reference(counting, scoring):
    # always: the original's stored answers (tests/golden/make_golden.py), with every restatement and every method as below
    # -- here score_points clusters the references itself, as the original did when the golden scores were made
    seqs = _seqs(counting)
    for k in (3, 4, 5, 6):
        want = counting["counts_k%d" % k]
        assert np.array_equal(c_oracle.count(counting["seq_bytes"], counting["seq_offsets"], k), want)
        for i, s in enumerate(seqs):
            assert np.array_equal(po.count_string_np(s, k), want[i])
            if len(s) <= 3001:
                assert np.array_equal(po.count_string(s, k), want[i])
    assert np.array_equal(po.normalize_counts(counting["counts_k4"]), counting["normalized_k4"], equal_nan=True)
    g, pos, neg = scoring
    pts = po.normalize_counts(g["query_counts"])
    for method in ("knn", "kmeans", "combo"):
        got = po.score_points(pts, pos, neg, method=method)
        assert np.max(np.abs(got - g["scores_" + method])) <= 1e-9, method
    if not ref_loader.reference_available():
        return
    # and, where the original scripts are installed (PHAMERS_REF), against them on fresh random inputs
    kmer, learning, phamer = ref_loader.load_reference()
    rng = np.random.default_rng(7)
    alphabet = np.frombuffer(b"ATGCATGCATGCATGCNatgcRY-", dtype=np.uint8)
    for k in (3, 4, 5, 6):
        for length in (0, 2, 5, 64, 700, 3001):
            s = rng.choice(alphabet, size=length).tobytes().decode("ascii")
            want = kmer.count_string(s, k)
            assert np.array_equal(po.count_string(s, k), want)
            assert np.array_equal(po.count_string_np(s, k), want)
            assert np.array_equal(c_oracle.count(np.frombuffer(s.encode(), dtype=np.uint8), [0, length], k)[0], want)
    counts = rng.integers(0, 50, size=(5, 256))
    assert np.array_equal(po.normalize_counts(counts), kmer.normalize_counts(counts))
    pos, neg, pts = (po.normalize_counts(rng.integers(1, 60, size=(n, 256))) for n in (120, 130, 40))
    for method in ("knn", "kmeans", "combo"):
        want = phamer.score_points(pts, pos, neg, method=method)
        got = po.score_points(pts, pos, neg, method=method)
        assert np.max(np.abs(got - want)) <= 1e-12

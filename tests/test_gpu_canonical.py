"""GPU checks of strand-independent scoring on canonical 4-mer features (136 bins): phm_canonical_fold against the oracle's fold,
the tensor-core road at width 136 against the exhaustive road and a float64 direct-difference oracle (neighbour rules (a)-(e) of
test_gpu_neighbors.py), the overflow roads, counts against features, the error bound, parity with the scikit-learn restatement,
and the point of the feature: a contig and its reverse complement get the same score and the same neighbours.
PHM_FUZZ_ROUNDS scales the randomised parts (default 4)."""
import os

import numpy as np
import pytest
import torch

from oracle import c_oracle
from oracle import phamers_oracle as po
from test_gpu_neighbors import _clear, _cuda, _oracle, _run, check_centroids, check_consistent, check_refs

pytestmark = pytest.mark.gpu
ROUNDS = int(os.environ.get("PHM_FUZZ_ROUNDS", "4"))
TOL = 1e-5
COMP = bytes.maketrans(b"ATGCN", b"TACGN")


@pytest.fixture(scope="module")
def canon(golden_dir):
    """Golden query counts and the shipped references, folded and normalised, with centroids fitted on the folded references."""
    from phamers_b200 import kmer, references
    g = np.load(os.path.join(golden_dir, "scoring_golden.npz"))
    _, pos_c, _, neg_c = references.load_reference_counts()
    n_ref = int(g["n_ref"])
    pos = kmer.normalize_counts(kmer.canonical_fold(pos_c[:n_ref], 4))
    neg = kmer.normalize_counts(kmer.canonical_fold(neg_c[:n_ref], 4))
    pts = kmer.normalize_counts(kmer.canonical_fold(g["query_counts"], 4))
    cp, cn = references.reference_centroids(pos, neg)
    return pos, neg, pts, cp, cn


def _draw(rng, base, n, depth):
    """n count rows from the composition families `base`; row totals vary from row to row, since with one common total the
    distances are quantised and truly tie (the roads may then order a tie differently)."""
    return np.stack([rng.multinomial(int(rng.integers(depth // 2, 2 * depth)), base[f]) for f in rng.integers(0, len(base), size=n)])


def _random_rows(rng, n, depth=3000, families=6):
    c = _draw(rng, rng.dirichlet(np.full(136, 0.5), size=families), n, depth).astype(np.float64)
    return c / c.sum(axis=1, keepdims=True)


def _random_seqs(rng, n, lo=2000, hi=9000):
    return [rng.choice(np.frombuffer(b"ATGC", dtype=np.uint8), size=int(rng.integers(lo, hi)),
                       p=np.array([1, 1, 1.6, 1.6]) / 5.2).tobytes().decode() for _ in range(n)]


def _device_seqs(seqs):
    blob = np.frombuffer("".join(seqs).encode(), dtype=np.uint8)
    off = np.concatenate(([0], np.cumsum([len(s) for s in seqs]))).astype(np.int64)
    d = torch.zeros(((len(blob) + 15) // 16 * 16 + 16,), dtype=torch.uint8, device="cuda")
    d[:len(blob)] = torch.from_numpy(blob.copy()).cuda()
    return d[:len(blob)], torch.from_numpy(off).cuda(), blob, off


# ---------------------------------------------------------------------------------------------------------------------
# fold
# ---------------------------------------------------------------------------------------------------------------------
def test_fold_bit_exact():
    from phamers_b200 import kmer, ops, references
    _, pos_c, _, neg_c = references.load_reference_counts()
    for c in (pos_c, neg_c):
        got = kmer.canonical_fold(c, 4)
        assert got.dtype == np.int64 and np.array_equal(got, po.canonical_fold(c, 4))
    rng = np.random.default_rng(4100)
    for round_ in range(ROUNDS):
        for k in range(1, 7):
            ints = rng.integers(0, 1 << 40, size=(int(rng.integers(1, 300)), 4 ** k))
            assert np.array_equal(kmer.canonical_fold(ints, k), po.canonical_fold(ints, k)), (round_, k)
            floats = rng.random((int(rng.integers(1, 300)), 4 ** k)) * 10.0 ** rng.integers(-3, 3)
            got = ops.canonical_fold_cuda(_cuda(floats), k).cpu().numpy()
            assert np.array_equal(got, po.canonical_fold(floats, k)), (round_, k)
            assert kmer.canonical_fold(floats, k).dtype == np.float64
    # the counter's canonical counts are the fold of its plain counts
    seqs = _random_seqs(rng, 200, 1, 3000)
    d_seq, d_off, _, _ = _device_seqs(seqs)
    for k in range(1, 7):
        plain, _ = ops.count_cuda(d_seq, d_off, k)
        canon, _ = ops.count_cuda(d_seq, d_off, k, canonical=True)      # counts of these contigs stay far below 2^31
        assert torch.equal(ops.canonical_fold_cuda(plain.to(torch.float64), k), canon.to(torch.float64)), k
    assert ops.canonical_fold_cuda(torch.zeros((0, 256), dtype=torch.float64, device="cuda"), 4).shape == (0, 136)


# ---------------------------------------------------------------------------------------------------------------------
# tensor-core road at width 136 against the exhaustive road
# ---------------------------------------------------------------------------------------------------------------------
def _hard_case(canon, rng, n_random=600):
    """Golden queries, random rows, queries sitting on references, references duplicated with the opposite label, NaN rows."""
    pos, neg, pts, cp, cn = canon
    pos, neg = pos.copy(), neg.copy()
    neg[5:10] = pos[20:25]                                              # negatives that duplicate positives
    X = np.vstack((pts, _random_rows(rng, n_random), pos[20:25], neg[40:45], pos[:3]))
    X[7] = np.nan
    X[len(pts) + 3] = np.nan
    return X, np.vstack((pos, neg)), len(pos), cp, cn


@pytest.mark.parametrize("k", [1, 3, 5])
def test_tensor_core_road_at_136(canon, k):
    X, R, n_pos, CP, CN = _hard_case(canon, np.random.default_rng(136 + k))
    args = (_cuda(X), _cuda(R), n_pos, _cuda(CP), _cuda(CN), k)
    tc, ex = _run(*args, path="tc"), _run(*args, path="exact")
    assert np.array_equal(tc[0], ex[0], equal_nan=True)                                   # votes
    for j in (1, 2):
        live = ~np.isnan(ex[j])
        assert np.array_equal(np.isnan(tc[j]), ~live)
        assert np.max(np.abs(tc[j][live] - ex[j][live])) <= 1e-12, j
    for out in (tc, ex):
        clear = check_refs(X, R, out[3], out[4], k)
        check_centroids(X, CP, CN, out[5], out[6])
        check_consistent(out, n_pos, k)
    live = ~np.isnan(X).any(axis=1)
    assert np.array_equal(tc[3][live][clear], ex[3][live][clear])
    on_ref = len(X) - 13                                                # the rows copied from references
    assert (tc[4][on_ref:on_ref + 10, 0] == 0.0).all()
    assert np.array_equal(tc[3][on_ref:on_ref + 5, 0], np.arange(20, 25))              # duplicate pair: the lower row
    assert (tc[3][7] == -1).all() and np.isnan(tc[0][7])


@pytest.mark.parametrize("n_rows", [300, 1000])                         # both sides of FB_BLOCKED_MIN (592)
def test_overflow_roads_at_136(canon, n_rows):
    from phamers_b200 import _lib
    X, R, n_pos, CP, CN = _hard_case(canon, np.random.default_rng(n_rows), n_random=1000)
    X = X[-n_rows:]
    X[3] = np.nan
    args = (_cuda(X), _cuda(R), n_pos, _cuda(CP), _cuda(CN), 3)
    base = _run(*args, path="tc")
    clear = check_refs(X, R, base[3], base[4], 3)
    live = ~np.isnan(X).any(axis=1)
    try:
        _lib.set_option("score_force_fallback", 1)
        for list_pass in (1, 0):
            _lib.set_option("score_list_pass", list_pass)
            road = _run(*args, path="tc")
            for a, b in zip(base[:3], road[:3]):
                assert np.array_equal(a, b, equal_nan=True), list_pass
            if list_pass or n_rows <= 592:
                assert np.array_equal(road[3][live], base[3][live]) and np.array_equal(road[4][live], base[4][live]), list_pass
            else:
                assert np.all(np.abs(road[4][live] - base[4][live]) <= 1e-13 * base[4][live]), list_pass
                assert np.array_equal(road[3][live][clear], base[3][live][clear]), list_pass
            assert np.array_equal(road[5], base[5]) and np.array_equal(road[6], base[6], equal_nan=True), list_pass
    finally:
        _lib.set_option("score_force_fallback", 0)
        _lib.set_option("score_list_pass", 1)


def test_counts_against_features_and_error_bound(canon):
    from phamers_b200 import _lib, ops
    pos, neg, _, cp, cn = canon
    rng = np.random.default_rng(2136)
    seqs = _random_seqs(rng, 3000) + [""]                               # the empty contig is a NaN row
    d_seq, d_off, _, _ = _device_seqs(seqs)
    counts, _ = ops.count_cuda(d_seq, d_off, 4, canonical=True)
    feats = ops.normalize_cuda(counts)
    R = _cuda(np.vstack((pos, neg)))
    for k in (1, 3, 5):
        f = _run(feats, R, len(pos), _cuda(cp), _cuda(cn), k, path="tc")
        c = _run(counts, R, len(pos), _cuda(cp), _cuda(cn), k)                # count rows take the tensor cores under "auto"
        for a, b in zip(f, c):
            assert np.array_equal(a, b, equal_nan=True), k
    try:
        _lib.set_option("score_stats", 1)
        ops.score_cuda(counts, R, len(pos), _cuda(cp), _cuda(cn), 3)
        stats = ops.score_stats()
    finally:
        _lib.set_option("score_stats", 0)
    assert 0.0 < stats["max_bound_usage"] <= 1.0, stats


def test_parity_with_scikit_learn_restatement(canon):
    """Folded golden queries scored by the library and by the oracle's scikit-learn score_points with the same centroids."""
    from phamers_b200 import phamer
    pos, neg, pts, cp, cn = canon
    got = phamer.score_points(pts, pos, neg)
    want = po.score_points(pts, pos, neg, centroids=(cp, cn))
    R = np.vstack((pos, neg))
    s_val, s_idx, _ = _oracle(pts, R, 4)
    keep = _clear(R, s_val, s_idx, duplicates_decide=False)            # scikit-learn orders near ties its own way
    assert keep.mean() > 0.9
    assert np.max(np.abs(got[keep] - want[keep])) <= TOL
    assert np.array_equal(np.sign(got[keep]), np.sign(want[keep]))


# ---------------------------------------------------------------------------------------------------------------------
# strand independence and the command line
# ---------------------------------------------------------------------------------------------------------------------
def _strand_fasta(path, rng, n):
    seqs, ids = [], []
    for i, s in enumerate(_random_seqs(rng, n, 5000, 20000)):
        b = bytearray(s.encode())
        for _ in range(3):                                              # N runs
            a, run = int(rng.integers(0, len(b) - 20)), int(rng.integers(1, 20))
            b[a:a + run] = b"N" * run
        fwd = bytes(b).decode()
        rc = fwd.encode().translate(COMP)[::-1].decode()
        seqs += [fwd, rc]
        ids += ["f%d" % i, "r%d" % i]
    with open(path, "w") as fh:
        for i, s in zip(ids, seqs):
            fh.write(">pair_ID_%s\n%s\n" % (i, "\n".join(s[j:j + 70] for j in range(0, len(s), 70))))
    return ids, seqs


def test_reverse_complements_score_the_same(tmp_path):
    from phamers_b200 import phamer, pipeline
    rng = np.random.default_rng(777)
    fasta = tmp_path / "pairs.fasta"
    ids, seqs = _strand_fasta(fasta, rng, 150)
    sc = phamer.main(["-fasta", str(fasta), "-out", str(tmp_path / "canon"), "-l", "0", "-equal", "-canonical", "-neighbors"])
    assert list(sc.data_ids) == ids
    assert np.array_equal(sc.scores[0::2], sc.scores[1::2])
    for a in (sc.neighbor_ids, sc.neighbor_labels, sc.neighbor_distances, sc.nearest_clusters, sc.nearest_cluster_distances):
        assert np.array_equal(a[0::2], a[1::2])
    # the counts cached next to the FASTA are plain counts, shared by both modes
    plain = phamer.main(["-fasta", str(fasta), "-out", str(tmp_path / "plain"), "-l", "0", "-equal"])
    assert (plain.scores[0::2] != plain.scores[1::2]).any()              # plain 4-mers do depend on the strand
    _, _, seq_blob, offsets = _device_seqs(seqs)
    scorer = pipeline.ContigScorer(canonical=True)
    host = scorer.score_host(seq_blob, offsets)
    assert np.array_equal(host[0::2], host[1::2])
    # the command line scores feature rows (exhaustive road at width 136), ContigScorer count rows (tensor-core road)
    assert np.max(np.abs(host - sc.scores)) <= 1e-12 and np.array_equal(np.sign(host), np.sign(sc.scores))
    assert np.array_equal(pipeline.ContigScorer().score_host(seq_blob, offsets), plain.scores)


def test_cli_canonical_against_oracle(tmp_path):
    from phamers_b200 import fileIO, phamer, references
    from test_gpu_cli import _write_fasta
    rng = np.random.default_rng(20261021)
    indir = tmp_path / "sample"
    indir.mkdir()
    lengths, seqs = _write_fasta(indir / "contigs.fasta", rng, 300)
    scorer = phamer.main(["-in", str(indir), "-out", str(tmp_path / "out"), "-equal", "-l", "5000", "-canonical"])
    blob = np.frombuffer("".join(seqs).encode(), dtype=np.uint8)
    offsets = np.concatenate(([0], np.cumsum([len(s) for s in seqs]))).astype(np.int64)
    keep = lengths >= 5000
    X = po.normalize_counts(po.canonical_fold(c_oracle.count(blob, offsets, 4)[keep], 4))
    pos, neg = references.load_reference_features(equalize=True, canonical=True)
    _, pos_c, _, neg_c = references.load_reference_counts()
    n = min(len(pos_c), len(neg_c))
    assert np.array_equal(pos, po.normalize_counts(po.canonical_fold(pos_c[:n], 4)))
    want = po.score_points(X, pos, neg, centroids=references.reference_centroids(pos, neg))
    by_id = fileIO.read_phamer_output(str(tmp_path / "out" / "phamer_scores.csv"))
    assert list(by_id) == [str(i) for i in np.nonzero(keep)[0]]
    got = np.array(list(by_id.values()))
    assert np.max(np.abs(got - want)) <= TOL and np.array_equal(np.sign(got), np.sign(want))
    assert "canonical_kmers:\tTrue" in open(tmp_path / "out" / "phamer_scores.csv").read()
    # the cached features are plain counts; a canonical-width features CSV is taken as it is
    _, cached = fileIO.read_feature_file(str(indir / "contigs_features.csv"))
    assert cached.shape == (300, 256)
    folded = tmp_path / "folded.csv"
    fileIO.save_counts(po.canonical_fold(cached, 4), np.arange(300), str(folded))
    again = phamer.main(["-features", str(folded), "-out", str(tmp_path / "out2"), "-equal", "-canonical"])
    assert np.array_equal(again.scores[keep], scorer.scores)


@pytest.mark.parametrize("round_", range(ROUNDS))
def test_random_rounds_at_136(round_):
    """Random reference sets and queries at width 136: tensor-core road (from counts) against the exhaustive road and the oracle."""
    rng = np.random.default_rng(36000 + round_)
    n_refs = int(rng.integers(50, 3000))
    n_pos = int(rng.integers(1, n_refs))
    depth = int(rng.choice([200, 3000, 50000]))
    fam = int(rng.integers(1, 12))
    base = rng.dirichlet(np.full(136, float(rng.choice([0.1, 0.5, 2.0]))), size=fam)
    ref_c, q_c = _draw(rng, base, n_refs, depth), _draw(rng, base, int(rng.integers(100, 2000)), depth)
    q_c[0] = 0
    R = ref_c / ref_c.sum(axis=1, keepdims=True)
    CP, CN = (_random_rows(rng, int(rng.integers(1, 40))) for _ in range(2))
    kn = int(rng.choice([1, 3, 5]))
    counts = torch.from_numpy(q_c.astype(np.int32)).cuda()
    from phamers_b200 import ops
    feats = ops.normalize_cuda(counts)
    X = feats.cpu().numpy()
    tc = _run(counts, _cuda(R), n_pos, _cuda(CP), _cuda(CN), kn, path="tc")
    ex = _run(feats, _cuda(R), n_pos, _cuda(CP), _cuda(CN), kn, path="exact")
    assert np.array_equal(tc[0], ex[0], equal_nan=True), round_
    for out in (tc, ex):
        clear = check_refs(X, R, out[3], out[4], kn, round_)
        check_centroids(X, CP, CN, out[5], out[6], round_)
        check_consistent(out, n_pos, kn, round_)
    live = ~np.isnan(X).any(axis=1)
    assert np.array_equal(tc[3][live][clear], ex[3][live][clear]), round_

"""GPU checks of the neighbour report (phm_score_neighbors / phm_score_counts_neighbors, ops.score_neighbors_cuda,
learning.kneighbors, phamer_scorer.score_neighbors, phamer -neighbors) against a float64 direct-difference oracle.

Index rules (the oracle sorts by distance, ties by lower index):
  (a) each returned distance equals the oracle's distance to the returned index within 1e-12 relative;
  (b) returned distances are non-decreasing;
  (c) the k-th returned distance is at most the oracle's k-th smallest x (1 + 1e-12): no closer reference was missed;
  (d) indices equal the oracle's wherever it has no near tie (relative gap <= 1e-12) among its first k + 1 distances;
  (e) bitwise-equal reference rows tie exactly and resolve to the lower index (they are not counted as near ties in (d)).
PHM_FUZZ_ROUNDS scales the randomised rounds (default 4)."""
import os

import numpy as np
import pytest
import torch

from oracle import c_oracle

pytestmark = pytest.mark.gpu
ROUNDS = int(os.environ.get("PHM_FUZZ_ROUNDS", "4"))


# ---------------------------------------------------------------------------------------------------------------------
# oracle and rules
# ---------------------------------------------------------------------------------------------------------------------
def _oracle(X, R, m, picks=None):
    """Direct-difference float64 distances of X's rows to R's rows (on the device, in chunks): the m smallest per row (stable: ties
    by lower index) and the distances at picks[n, j] (>= 0)."""
    Xt, Rt = torch.from_numpy(np.ascontiguousarray(X)).cuda(), torch.from_numpy(np.ascontiguousarray(R)).cuda()
    if picks is None:
        picks = np.zeros((X.shape[0], 1), dtype=np.int64)
    pk = torch.from_numpy(np.ascontiguousarray(picks)).cuda()
    step = max(1, int(1.5e9 // (R.shape[0] * R.shape[1] * 8)))
    vals, idxs, at = [], [], []
    for lo in range(0, X.shape[0], step):
        d = torch.sqrt(((Xt[lo:lo + step, None, :] - Rt[None]) ** 2).sum(-1))
        s, o = torch.sort(d, dim=1, stable=True)
        vals.append(s[:, :m].cpu())
        idxs.append(o[:, :m].cpu())
        at.append(torch.gather(d, 1, pk[lo:lo + step]).cpu())
    cat = lambda parts, w, dt: torch.cat(parts).numpy() if parts else np.zeros((0, w), dtype=dt)
    return cat(vals, m, np.float64), cat(idxs, m, np.int64), cat(at, picks.shape[1], np.float64)


def _clear(R, s_val, s_idx, duplicates_decide=True):
    """Rows whose oracle order has no near tie among the listed distances.  Ties of bitwise-equal rows are exact and go to the lower
    index (rule (e)), so they count as decided unless duplicates_decide is False (for a library without that rule)."""
    if s_val.shape[1] < 2:
        return np.ones(s_val.shape[0], dtype=bool)
    gap = s_val[:, 1:] - s_val[:, :-1]
    same = (R[s_idx[:, 1:]] == R[s_idx[:, :-1]]).all(axis=-1) if duplicates_decide else np.zeros(gap.shape, dtype=bool)
    return ~((gap <= 1e-12 * s_val[:, 1:]) & ~same).any(axis=1)


def check_refs(X, R, idx, dist, k, tag=""):
    live = ~np.isnan(X).any(axis=1)
    assert idx.shape == dist.shape == (X.shape[0], k), tag
    assert (idx[~live] == -1).all() and np.isnan(dist[~live]).all(), tag
    I, D = idx[live], dist[live]
    assert ((I >= 0) & (I < R.shape[0])).all(), tag
    s_val, s_idx, at = _oracle(X[live], R, min(k + 1, R.shape[0]), I)
    assert np.all(np.abs(D - at) <= 1e-12 * at), tag                                   # (a)
    assert np.all(np.diff(D, axis=1) >= 0), tag                                         # (b)
    assert np.all(D[:, k - 1] <= s_val[:, k - 1] * (1 + 1e-12)), tag                     # (c)
    clear = _clear(R, s_val, s_idx)
    assert np.array_equal(I[clear], s_idx[clear, :k]), tag                              # (d), (e)
    return clear


def check_centroids(X, CP, CN, ci, cd, tag=""):
    live = ~np.isnan(X).any(axis=1)
    assert (ci[~live] == -1).all() and np.isnan(cd[~live]).all(), tag
    for c, C in enumerate((CP, CN)):
        if C.shape[0] == 0:
            assert (ci[:, c] == -1).all() and np.isnan(cd[:, c]).all(), tag
            continue
        I, D = ci[live, c], cd[live, c]
        assert ((I >= 0) & (I < C.shape[0])).all(), tag
        s_val, s_idx, at = _oracle(X[live], C, min(2, C.shape[0]), I[:, None])
        assert np.all(np.abs(D - at[:, 0]) <= 1e-12 * at[:, 0]), tag
        assert np.all(D <= s_val[:, 0] * (1 + 1e-12)), tag
        clear = _clear(C, s_val, s_idx)
        assert np.array_equal(I[clear], s_idx[clear, 0]), tag


def check_consistent(out, n_pos, k, tag=""):
    """The reported rows give the reported scores: the vote of their labels, and tanh((cd[1] - cd[0]) / (cd[0] + cd[1]))."""
    knn, km, _, idx, _, _, cd = out
    live = ~np.isnan(knn)
    pos = (idx[live] < n_pos).sum(axis=1)
    assert np.array_equal(np.where(2 * pos > k, 1.0, -1.0), knn[live]), tag
    if not np.isnan(cd[live]).any():
        want = np.tanh((cd[live, 1] - cd[live, 0]) / (cd[live, 0] + cd[live, 1]))
        assert np.max(np.abs(want - km[live]), initial=0.0) <= 4e-16, tag                 # device tanh vs numpy tanh: last bit


def _np(out):
    return [t.cpu().numpy() for t in out]


def _run(points, refs, n_pos, cp, cn, k, path="auto"):
    """(scores of score_cuda, the seven arrays of score_neighbors_cuda) on one road; the scores must be bit-identical."""
    from phamers_b200 import ops
    try:
        ops.set_score_path(path)
        plain = _np(ops.score_cuda(points, refs, n_pos, cp, cn, k))
        out = _np(ops.score_neighbors_cuda(points, refs, n_pos, cp, cn, k))
    finally:
        ops.set_score_path("auto")
    for a, b in zip(plain, out[:3]):
        assert np.array_equal(a, b, equal_nan=True)
    return out


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(scope="module")
def golden(golden_dir):
    from phamers_b200 import kmer, references
    g = np.load(os.path.join(golden_dir, "scoring_golden.npz"))
    _, pos_c, _, neg_c = references.load_reference_counts()
    n_ref = int(g["n_ref"])
    pos, neg = kmer.normalize_counts(pos_c[:n_ref]), kmer.normalize_counts(neg_c[:n_ref])
    return g, pos, neg, kmer.normalize_counts(g["query_counts"])


def _random_case(rng, n_pts, n_refs, dim=256, n_cp=20, n_cn=17, depth=3000):
    base = rng.dirichlet(np.full(dim, 0.5), size=6)
    def sample(n):
        return np.stack([rng.multinomial(depth, base[f]) for f in rng.integers(0, 6, size=n)]).astype(np.float64)
    norm = lambda c: c / np.maximum(c.sum(axis=1, keepdims=True), 1)
    return norm(sample(n_pts)), norm(sample(n_refs)), norm(sample(n_cp)), norm(sample(n_cn))


# ---------------------------------------------------------------------------------------------------------------------
# 1. golden queries
# ---------------------------------------------------------------------------------------------------------------------
def test_golden_neighbors(golden, monkeypatch):
    from phamers_b200 import phamer, references
    g, pos, neg, pts = golden
    R = np.vstack((pos, neg))
    CP, CN = g["centroids_pos"], g["centroids_neg"]
    out = _run(_cuda(pts), _cuda(R), len(pos), _cuda(CP), _cuda(CN), 3)
    check_refs(pts, R, out[3], out[4], 3)
    check_centroids(pts, CP, CN, out[5], out[6])
    check_consistent(out, len(pos), 3)
    assert np.array_equal(out[0], g["scores_knn"])
    monkeypatch.setattr(references, "reference_centroids", lambda p, n, k=86: (CP, CN))
    for j, method in enumerate(("knn", "kmeans", "combo")):
        assert np.array_equal(out[j], phamer.score_points(pts, pos, neg, method=method), equal_nan=True), method


# ---------------------------------------------------------------------------------------------------------------------
# 2. / 3. tensor-core road against the exhaustive road; the exhaustive kernel's own shapes
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 3, 5])
def test_tensor_core_road_against_exhaustive_road(golden, k):
    g, pos, neg, pts = golden
    R = np.vstack((pos, neg))
    CP, CN = g["centroids_pos"], g["centroids_neg"]
    rng = np.random.default_rng(10 + k)
    X = np.vstack((pts, _random_case(rng, 500, 1)[0]))
    args = (_cuda(X), _cuda(R), len(pos), _cuda(CP), _cuda(CN), k)
    tc, ex = _run(*args, path="tc"), _run(*args, path="exact")
    for out in (tc, ex):
        clear = check_refs(X, R, out[3], out[4], k)
        check_centroids(X, CP, CN, out[5], out[6])
        check_consistent(out, len(pos), k)
    assert np.array_equal(tc[3][clear], ex[3][clear])
    assert np.all(np.abs(tc[4] - ex[4]) <= 1e-12 * ex[4])


@pytest.mark.parametrize("k,dim", [(7, 256), (15, 256), (3, 136), (5, 1024), (15, 136)])
def test_exhaustive_kernel_shapes(k, dim):
    rng = np.random.default_rng(k * 1000 + dim)
    X, R, CP, CN = _random_case(rng, 150, 700, dim=dim)
    X[5] = R[17]                                                       # a query on a reference: distance 0
    X[9] = np.nan
    out = _run(_cuda(X), _cuda(R), 300, _cuda(CP), _cuda(CN), k)
    check_refs(X, R, out[3], out[4], k)
    assert out[3][5, 0] == 17 and out[4][5, 0] == 0.0
    check_centroids(X, CP, CN, out[5], out[6])
    check_consistent(out, 300, k)
    # one empty centroid set: that class reports -1 / NaN, the other its nearest
    from phamers_b200 import ops
    one = _np(ops.score_neighbors_cuda(_cuda(X), _cuda(R), 300, _cuda(CP), _cuda(CN[:0]), k))
    check_centroids(X, CP, CN[:0], one[5], one[6])
    assert np.array_equal(one[3], out[3])


# ---------------------------------------------------------------------------------------------------------------------
# 4. every overflow road gives the default road's neighbours
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_rows", [300, 1000])                         # both sides of FB_BLOCKED_MIN (592)
def test_overflow_roads(golden, n_rows):
    from phamers_b200 import _lib
    g, pos, neg, pts = golden
    R = np.vstack((pos, neg))
    CP, CN = g["centroids_pos"], g["centroids_neg"]
    rng = np.random.default_rng(n_rows)
    X = np.vstack((pts, _random_case(rng, n_rows, 1)[0]))[:n_rows]
    X[3] = np.nan
    args = (_cuda(X), _cuda(R), len(pos), _cuda(CP), _cuda(CN), 3)
    base = _run(*args)
    clear = check_refs(X, R, base[3], base[4], 3)
    try:
        _lib.set_option("score_force_fallback", 1)
        for list_pass in (1, 0):
            _lib.set_option("score_list_pass", list_pass)
            road = _run(*args)
            for a, b in zip(base[:3], road[:3]):
                assert np.array_equal(a, b, equal_nan=True), list_pass
            live = ~np.isnan(X).any(axis=1)
            if list_pass or n_rows <= 592:
                # list pass and sliced exhaustive kernel: the default road's arithmetic and order, bit for bit
                assert np.array_equal(road[3][live], base[3][live]), list_pass
                assert np.array_equal(road[4][live], base[4][live]), list_pass
            else:
                # blocked exhaustive kernel: its own summation order (last bits of the distances)
                assert np.all(np.abs(road[4][live] - base[4][live]) <= 1e-13 * base[4][live]), list_pass
                assert np.array_equal(road[3][live][clear], base[3][live][clear]), list_pass
            assert np.array_equal(road[5], base[5]) and np.array_equal(road[6], base[6], equal_nan=True), list_pass
            check_refs(X, R, road[3], road[4], 3, tag=list_pass)
    finally:
        _lib.set_option("score_force_fallback", 0)
        _lib.set_option("score_list_pass", 1)


# ---------------------------------------------------------------------------------------------------------------------
# 5. / 6. / 7. duplicates of opposite labels, queries on references, NaN rows, counts against features
# ---------------------------------------------------------------------------------------------------------------------
def test_duplicates_queries_on_references_nan_rows_and_counts():
    from phamers_b200 import ops
    rng = np.random.default_rng(77)
    base = rng.dirichlet(np.full(256, 0.7), size=5)
    ref_c = np.stack([rng.multinomial(5000, base[i % 5]) for i in range(400)])
    ref_c[300:310] = ref_c[10:20]                                       # negatives that duplicate positives (labels differ)
    ref_c[40:45] = ref_c[30:35]                                         # duplicates inside one class
    q_c = np.stack([rng.multinomial(4000, base[i % 5]) for i in range(700)])
    q_c[:20] = ref_c[300:320]                                           # queries sitting exactly on references
    q_c[25:30] = ref_c[30:35]
    q_c[50] = 0                                                         # an empty contig -> NaN row
    R = ref_c / ref_c.sum(axis=1, keepdims=True)
    cp_c, cn_c = rng.integers(1, 50, size=(12, 256)), rng.integers(1, 50, size=(9, 256))
    cn_c[4] = cn_c[2]                                                   # tied centroids: the first one is reported
    CP, CN = cp_c / cp_c.sum(axis=1, keepdims=True), cn_c / cn_c.sum(axis=1, keepdims=True)
    counts = torch.from_numpy(q_c.astype(np.int32)).cuda()
    feats = ops.normalize_cuda(counts)
    X = feats.cpu().numpy()
    for k in (1, 3, 5):
        f = _run(feats, _cuda(R), 200, _cuda(CP), _cuda(CN), k)
        c = _run(counts, _cuda(R), 200, _cuda(CP), _cuda(CN), k)
        for a, b in zip(f, c):                                          # 7: counts give the features' answer bit for bit
            assert np.array_equal(a, b, equal_nan=True), k
        check_refs(X, R, f[3], f[4], k, tag=k)
        check_centroids(X, CP, CN, f[5], f[6], tag=k)
        check_consistent(f, 200, k, tag=k)
        assert (f[4][:20, 0] == 0.0).all() and np.array_equal(f[3][:10, 0], np.arange(10, 20))    # lower index of the duplicate
        assert np.array_equal(f[3][10:20, 0], np.arange(310, 320))
        assert np.array_equal(f[3][25:30, 0], np.arange(30, 35))
        assert (f[3][50] == -1).all() and np.isnan(f[4][50]).all() and (f[5][50] == -1).all() and np.isnan(f[6][50]).all()
        assert not (f[5][:, 1] == 4).any()                                # centroid 4 ties centroid 2 bit for bit


# ---------------------------------------------------------------------------------------------------------------------
# 8. enlarged reference set
# ---------------------------------------------------------------------------------------------------------------------
def test_enlarged_references(golden):
    from tools import workloads
    g, pos, neg, pts = golden
    refs, n_pos = workloads.enlarged_references(pos, neg, 120000)
    R = refs.cpu().numpy()
    rng = np.random.default_rng(8)
    X = np.vstack((pts, R[rng.integers(0, len(R), size=200)], _random_case(rng, 1500, 1)[0]))
    CP, CN = g["centroids_pos"], g["centroids_neg"]
    args = (_cuda(X), refs, n_pos, _cuda(CP), _cuda(CN), 3)
    tc, ex = _run(*args), _run(*args, path="exact")
    clear = check_refs(X, R, tc[3], tc[4], 3)
    check_refs(X, R, ex[3], ex[4], 3)
    assert np.array_equal(tc[3][clear], ex[3][clear])
    check_centroids(X, CP, CN, tc[5], tc[6])
    check_consistent(tc, n_pos, 3)


# ---------------------------------------------------------------------------------------------------------------------
# 9. learning.kneighbors against scikit-learn
# ---------------------------------------------------------------------------------------------------------------------
def test_learning_kneighbors_against_scikit_learn(golden):
    from sklearn.neighbors import NearestNeighbors
    from phamers_b200 import learning
    _, pos, neg, pts = golden
    R = np.vstack((pos, neg))[np.random.default_rng(9).permutation(len(pos) + len(neg))]
    for k in (1, 4, 15):
        dist, idx = learning.kneighbors(pts, R, k=k)
        want_d, want_i = NearestNeighbors(n_neighbors=k, algorithm="brute").fit(R).kneighbors(pts)
        assert dist.shape == idx.shape == (len(pts), k) and idx.dtype == np.int64
        # scikit-learn forms |x|^2 - 2 x.y + |y|^2: a rounding error e of the squared distance moves the distance by at most
        # min(e / d, sqrt(e)), which matters for a query sitting on a reference (d = 0 here, about 1e-9 there)
        err = 4e-15 * ((pts ** 2).sum(axis=1)[:, None] + (R[want_i] ** 2).sum(axis=2))
        slack = np.minimum(err / np.maximum(want_d, 1e-300), np.sqrt(err))
        assert np.all(np.abs(dist - want_d) <= 1e-12 * want_d + slack), k
        check_refs(pts, R, idx, dist, k)
        s_val, s_idx, _ = _oracle(pts, R, min(k + 1, R.shape[0]))
        clear = _clear(R, s_val, s_idx, duplicates_decide=False)     # scikit-learn orders exact ties arbitrarily
        assert np.array_equal(idx[clear], want_i[clear]), k


# ---------------------------------------------------------------------------------------------------------------------
# 10. the command line
# ---------------------------------------------------------------------------------------------------------------------
def test_cli_writes_neighbor_file(tmp_path):
    from phamers_b200 import fileIO, phamer, references
    from test_gpu_cli import _write_fasta            # tests/ is on sys.path under pytest
    rng = np.random.default_rng(20260101)
    indir = tmp_path / "sample"
    indir.mkdir()
    lengths, seqs = _write_fasta(indir / "contigs.fasta", rng, 300)
    out = tmp_path / "nb"                                                # the score file's header names the output directory
    phamer.main(["-in", str(indir), "-out", str(out), "-equal", "-l", "5000"])
    plain = open(out / "phamer_scores.csv", "rb").read()
    scorer = phamer.main(["-in", str(indir), "-out", str(out), "-equal", "-l", "5000", "-neighbors"])
    assert open(out / "phamer_scores.csv", "rb").read() == plain
    ids, ref_ids, labels, dist, clusters, cdist = fileIO.read_phamer_neighbors(str(tmp_path / "nb" / "phamer_neighbors.csv"))
    assert list(ids) == list(fileIO.read_phamer_output(str(tmp_path / "nb" / "phamer_scores.csv")))
    # oracle: the contigs counted by the C restatement, distances to the equalised shipped references and their centroids
    blob = np.frombuffer("".join(seqs).encode(), dtype=np.uint8)
    offsets = np.concatenate(([0], np.cumsum([len(s) for s in seqs]))).astype(np.int64)
    counts = c_oracle.count(blob, offsets, 4)[lengths >= 5000]
    X = counts / counts.sum(axis=1, keepdims=True)
    pid, pos_c, nid, neg_c = references.load_reference_counts()
    n = min(len(pos_c), len(neg_c))
    pos, neg = references.load_reference_features(equalize=True)
    R = np.vstack((pos, neg))
    all_ids = np.concatenate((pid[:n], nid[:n])).astype(str)
    s_val, s_idx, _ = _oracle(X, R, 4)
    assert np.all(np.abs(dist - s_val[:, :3]) <= 1e-12 * s_val[:, :3])
    clear = _clear(R, s_val, s_idx)
    assert clear.mean() > 0.9
    assert np.array_equal(ref_ids[clear], all_ids[s_idx[clear, :3]])
    assert np.array_equal(labels[clear], (s_idx[clear, :3] < n).astype(np.int64))
    assert np.array_equal(dist, scorer.neighbor_distances) and np.array_equal(clusters, scorer.nearest_clusters)
    CP, CN = references.reference_centroids(pos, neg)
    check_centroids(X, CP, CN, clusters, cdist)


# ---------------------------------------------------------------------------------------------------------------------
# 11. randomised rounds
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("round_", range(ROUNDS))
def test_random_rounds_neighbors(round_):
    """Random shapes and composition families (tests/test_gpu_fuzz.py's generator): the tensor-core neighbour road against the
    exhaustive road and the oracle."""
    from phamers_b200 import kmer, ops
    from test_gpu_fuzz import _scoring_case
    rng = np.random.default_rng(55000 + round_)
    ref_counts, n_pos, q_counts, cen_p, cen_n, kn, tag = _scoring_case(rng)
    R, CP, CN = kmer.normalize_counts(ref_counts), kmer.normalize_counts(cen_p), kmer.normalize_counts(cen_n)
    counts = torch.from_numpy(q_counts.astype(np.int32)).cuda()
    feats = ops.normalize_cuda(counts)
    X = feats.cpu().numpy()
    tc = _run(counts, _cuda(R), n_pos, _cuda(CP), _cuda(CN), kn, path="tc")
    ex = _run(feats, _cuda(R), n_pos, _cuda(CP), _cuda(CN), kn, path="exact")
    tag = str(round_) + " " + tag
    for out in (tc, ex):
        clear = check_refs(X, R, out[3], out[4], kn, tag)
        check_centroids(X, CP, CN, out[5], out[6], tag)
        check_consistent(out, n_pos, kn, tag)
    live = ~np.isnan(X).any(axis=1)
    assert np.array_equal(tc[3][live][clear], ex[3][live][clear]), tag

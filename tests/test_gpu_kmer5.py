"""GPU checks of scoring 5-mer count rows on the tensor cores (1024 plain and 512 canonical bins): the tensor-core road against the
exhaustive float64 road on the same rows (votes identical, scores within 1e-12, outside exact rational ties), the neighbour
report against a direct-difference oracle (rules (a)-(e) of test_gpu_neighbors.py), the overflow roads (list pass and both
exhaustive fallbacks), the proven error bound, strand independence of canonical 5-mers, ContigScorer(kmer_length=5) against
phamer_scorer, and phm_score on float64 rows keeping the exhaustive kernel at these widths.  Every row is counted on the device
from synthetic sequences."""
import numpy as np
import pytest
import torch

from test_gpu_neighbors import _cuda, _run, check_centroids, check_consistent, check_refs

pytestmark = pytest.mark.gpu
COMP = bytes.maketrans(b"ATGCN", b"TACGN")
MODES = [(False, 1024), (True, 512)]
MODE_IDS = ["plain1024", "canonical512"]


def _family(rng):
    """A composition family: 48 random 6-base words with Dirichlet weights, so families differ in their 5-mer spectra."""
    return rng.integers(0, 4, size=(48, 6)), rng.dirichlet(np.full(48, 0.4))


def _seq(rng, fam, length):
    words, w = fam
    s = words[rng.choice(len(w), size=length // 6 + 1, p=w)].ravel()[:length]
    mut = rng.random(length) < 0.08                                    # every 5-mer can occur
    s[mut] = rng.integers(0, 4, size=int(mut.sum()))
    return np.frombuffer(b"ATGC", dtype=np.uint8)[s].tobytes().decode()


def _seqs(rng, fams, n, lo, hi):
    return [_seq(rng, fams[int(rng.integers(len(fams)))], int(rng.integers(lo, hi))) for _ in range(n)]


def _device_seqs(seqs):
    blob = np.frombuffer("".join(seqs).encode(), dtype=np.uint8)
    off = np.concatenate(([0], np.cumsum([len(s) for s in seqs]))).astype(np.int64)
    d = torch.zeros(((len(blob) + 15) // 16 * 16 + 16,), dtype=torch.uint8, device="cuda")
    d[:len(blob)] = torch.from_numpy(blob.copy()).cuda()
    return d[:len(blob)], torch.from_numpy(off).cuda()


def _count(seqs, canonical):
    from phamers_b200 import ops
    d_seq, d_off = _device_seqs(seqs)
    counts, _ = ops.count_cuda(d_seq, d_off, 5, canonical=canonical)
    return counts


def _centroids(rows, rng, n):
    """Centroids: means of random groups of rows (exact float64 rows of the right width; k-means is not what is tested here)."""
    groups = rng.integers(0, n, size=rows.shape[0])
    return np.stack([rows[groups == g].mean(axis=0) if (groups == g).any() else rows[g] for g in range(n)])


@pytest.fixture(scope="module", params=MODES, ids=MODE_IDS)
def case(request):
    """(canonical, width, query counts int32 on the device, references float64, n_positive, centroids +, centroids -, fams).
    Queries: deep and shallow contigs, count rows of references (queries sitting on references), empty contigs (NaN rows).
    References: 320 positives and 320 negatives of 8 families; negatives 5..9 duplicate positives 20..24 (opposite labels)."""
    from phamers_b200 import kmer
    canonical, width = request.param
    rng = np.random.default_rng(5000 + width)
    fams = [_family(rng) for _ in range(8)]
    ref_c = _count(_seqs(rng, fams[:4], 320, 3000, 30000) + _seqs(rng, fams[3:], 320, 3000, 30000), canonical).cpu().numpy()
    ref_c[320 + 5:320 + 10] = ref_c[20:25]
    R = kmer.normalize_counts(ref_c.astype(np.int64))
    q = _count(_seqs(rng, fams, 500, 2000, 40000) + _seqs(rng, fams, 150, 20, 400) + ["", "ACG"], canonical).cpu().numpy()
    q = np.vstack((q, ref_c[20:25], ref_c[320 + 40:320 + 45], ref_c[:3]))
    q[7] = 0
    assert q.shape[1] == width
    CP, CN = _centroids(R[:320], rng, 9), _centroids(R[320:], rng, 7)
    return canonical, width, torch.from_numpy(q.astype(np.int32)).cuda(), R, 320, CP, CN, fams


def _decided(X, R, k):
    """Rows whose k-th and (k+1)-th nearest references are not an exact (rational) tie between distinct rows: the vote of such a
    row depends on the order of the float64 additions, which differs between the roads (as in test_gpu_fuzz.py)."""
    live = ~np.isnan(X[:, 0])
    d2 = (X[live] ** 2).sum(axis=1)[:, None] + (R ** 2).sum(axis=1)[None, :] - 2.0 * X[live] @ R.T
    order = np.argsort(d2, axis=1, kind="stable")
    decided = np.ones(len(X), dtype=bool)
    rows = np.arange(order.shape[0])
    a, b = order[:, k - 1], order[:, k]
    close = np.abs(d2[rows, b] - d2[rows, a]) <= 1e-10 * (np.abs(d2[rows, a]) + 1e-30)
    same_row = (R[a] == R[b]).all(axis=1)
    decided[np.flatnonzero(live)[close & ~same_row]] = False
    return decided


@pytest.mark.parametrize("k", [1, 3, 5])
def test_tensor_cores_against_exhaustive(case, k):
    from phamers_b200 import ops
    _, width, counts, R, n_pos, CP, CN, _ = case
    feats = ops.normalize_cuda(counts)
    X = feats.cpu().numpy()
    refs = (_cuda(R), n_pos, _cuda(CP), _cuda(CN), k)
    tc = _run(counts, *refs)                                            # count rows take the tensor cores under "auto"
    ex = _run(feats, *refs, path="exact")
    decided = _decided(X, R, k)
    assert decided.mean() > 0.9
    assert np.array_equal(tc[0][decided], ex[0][decided], equal_nan=True)                  # votes
    live = ~np.isnan(X[:, 0])
    assert np.array_equal(np.isnan(tc[1]), ~live) and np.array_equal(np.isnan(ex[1]), ~live)
    assert np.max(np.abs(tc[1][live] - ex[1][live])) <= 1e-12
    ok = live & decided
    assert np.max(np.abs(tc[2][ok] - ex[2][ok])) <= 1e-12
    for out in (tc, ex):
        clear = check_refs(X, R, out[3], out[4], k, width)
        check_centroids(X, CP, CN, out[5], out[6], width)
        check_consistent(out, n_pos, k, width)
    assert np.array_equal(tc[3][live][clear], ex[3][live][clear])
    on_ref = len(X) - 13                                                # the rows copied from references
    assert (tc[4][on_ref:on_ref + 13, 0] == 0.0).all()
    assert np.array_equal(tc[3][on_ref:on_ref + 5, 0], np.arange(20, 25))                  # duplicate pair: the lower row
    assert np.array_equal(tc[3][on_ref + 5:on_ref + 10, 0], np.arange(320 + 40, 320 + 45))
    for r in (7, len(X) - 15):                                          # zero-count rows: NaN scores, -1 / NaN neighbours
        assert np.isnan(tc[0][r]) and np.isnan(tc[2][r]) and (tc[3][r] == -1).all() and (tc[5][r] == -1).all()
        assert np.isnan(tc[4][r]).all() and np.isnan(tc[6][r]).all()


@pytest.mark.parametrize("n_rows", [300, 661])                          # both sides of FB_BLOCKED_MIN (592)
def test_overflow_roads(case, n_rows):
    from phamers_b200 import _lib, ops
    _, width, counts, R, n_pos, CP, CN, _ = case
    counts = counts[-n_rows:].contiguous()
    X = ops.normalize_cuda(counts).cpu().numpy()
    live = ~np.isnan(X[:, 0])
    args = (counts, _cuda(R), n_pos, _cuda(CP), _cuda(CN))
    for k in (1, 3, 5):
        base = _run(*args, k)
        clear = check_refs(X, R, base[3], base[4], k, width)
        try:
            _lib.set_option("score_force_fallback", 1)
            for list_pass in (1, 0):
                _lib.set_option("score_list_pass", list_pass)
                road = _run(*args, k)
                tag = (width, n_rows, k, list_pass)
                for a, b in zip(base[:3], road[:3]):
                    assert np.array_equal(a, b, equal_nan=True), tag
                if list_pass or n_rows <= 592:
                    assert np.array_equal(road[3][live], base[3][live]) and np.array_equal(road[4][live], base[4][live]), tag
                else:                                                   # the blocked kernel orders by its own distance sum
                    assert np.all(np.abs(road[4][live] - base[4][live]) <= 1e-13 * base[4][live]), tag
                    assert np.array_equal(road[3][live][clear], base[3][live][clear]), tag
                assert np.array_equal(road[5], base[5]) and np.array_equal(road[6], base[6], equal_nan=True), tag
                if not list_pass:
                    assert ops.score_stats()["fallback_rows"] == int(live.sum()), tag
        finally:
            _lib.set_option("score_force_fallback", 0)
            _lib.set_option("score_list_pass", 1)


def test_error_bound(case):
    from phamers_b200 import _lib, ops
    _, _, counts, R, n_pos, CP, CN, _ = case
    try:
        _lib.set_option("score_stats", 1)
        for k in (1, 3, 5):
            ops.score_cuda(counts, _cuda(R), n_pos, _cuda(CP), _cuda(CN), k)
            stats = ops.score_stats()
            assert 0.0 < stats["max_bound_usage"] <= 1.0, (k, stats)
    finally:
        _lib.set_option("score_stats", 0)


def test_float64_rows_keep_the_exhaustive_kernel(case):
    """phm_score on feature rows at 512 / 1024 under "auto" is the exhaustive kernel, bit for bit, as before this road existed."""
    from phamers_b200 import ops
    _, _, counts, R, n_pos, CP, CN, _ = case
    feats = ops.normalize_cuda(counts)
    for k in (1, 3, 5):
        auto = _run(feats, _cuda(R), n_pos, _cuda(CP), _cuda(CN), k)
        exact = _run(feats, _cuda(R), n_pos, _cuda(CP), _cuda(CN), k, path="exact")
        for a, b in zip(auto, exact):
            assert np.array_equal(a, b, equal_nan=True), k


def test_canonical_reverse_complements_score_the_same():
    from phamers_b200 import kmer, ops
    rng = np.random.default_rng(5512)
    fams = [_family(rng) for _ in range(6)]
    R = kmer.normalize_counts(_count(_seqs(rng, fams, 400, 3000, 20000), True).cpu().numpy().astype(np.int64))
    fwd = _seqs(rng, fams, 300, 200, 20000)
    both = []
    for s in fwd:
        both += [s, s.encode().translate(COMP)[::-1].decode()]
    counts = _count(both, True)
    CP, CN = _centroids(R[:200], rng, 5), _centroids(R[200:], rng, 6)
    for k in (1, 3, 5):
        out = _run(counts, _cuda(R), 200, _cuda(CP), _cuda(CN), k)
        for a in out:
            assert np.array_equal(a[0::2], a[1::2], equal_nan=True), k
    plain = _count(both, False).cpu().numpy()
    assert (plain[0::2] != plain[1::2]).any()                           # plain 5-mers do depend on the strand


def _write_fasta(path, seqs):
    with open(path, "w") as fh:
        for i, s in enumerate(seqs):
            fh.write(">contig_ID_%d\n%s\n" % (i, "\n".join(s[j:j + 70] for j in range(0, len(s), 70))))


def test_contig_scorer_against_phamer_scorer(case, tmp_path):
    """ContigScorer(kmer_length=5) scores count rows on the tensor cores; phamer_scorer at k = 5 scores feature rows on the exhaustive
    kernel.  Same references, centroids and method: the same scores outside exact ties."""
    from phamers_b200 import kmer, phamer, pipeline, references
    canonical, width, _, R, n_pos, _, _, fams = case
    rng = np.random.default_rng(width + 77)
    seqs = _seqs(rng, fams, 200, 500, 20000) + [""]
    fasta = tmp_path / "k5.fasta"
    _write_fasta(fasta, seqs)
    pos, neg = R[:n_pos], R[n_pos:]
    cents = references.reference_centroids(pos, neg, 8)
    scorer = pipeline.ContigScorer(pos, neg, k_clusters=8, kmer_length=5, centroids=cents, canonical=canonical)
    ps = phamer.phamer_scorer()
    ps.kmer_length, ps.canonical, ps.k_clusters, ps.fasta_file = 5, canonical, 8, str(fasta)
    ps.positive_data, ps.negative_data = pos, neg
    ps.load_data(length_requirement=0)
    assert ps.data_points.shape == (len(seqs), width)
    decided = _decided(ps.data_points, R, 3)
    for method in ("combo", "knn", "kmeans"):
        ids, got = scorer.score_fasta(str(fasta), method=method)
        ps.scoring_method = method
        want = ps.score_points()
        assert list(ids) == [str(i) for i in range(len(seqs))]
        ok = decided & ~np.isnan(want)
        assert np.array_equal(np.isnan(got), np.isnan(want)), method
        assert np.max(np.abs(got[ok] - want[ok])) <= 1e-12, method
    blob = np.frombuffer("".join(seqs).encode(), dtype=np.uint8).copy()
    offsets = np.concatenate(([0], np.cumsum([len(s) for s in seqs]))).astype(np.int64)
    scorer.HOST_CHUNKS, scorer.HOST_CHUNK_MIN_BASES = 4, 100000
    host = scorer.score_host(blob, offsets)
    d_seq, d_off = _device_seqs(seqs)
    counts, dev = scorer.score_device(d_seq, d_off)
    assert counts.shape == (len(seqs), width)
    assert np.array_equal(host, dev.cpu().numpy(), equal_nan=True)
    assert np.array_equal(counts.cpu().numpy(), kmer.count(seqs, 5) if not canonical else kmer.canonical_fold(kmer.count(seqs, 5), 5))

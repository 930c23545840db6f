"""GPU checks of sliding-window scoring: window counts bit for bit against the C oracle on the window slices materialised on the host
(plain and canonical, k = 1..6, tiled windows, N / lower-case runs on window edges, 16- and 512-byte boundaries), slicing, scores
against score_cuda on the same rows and against the oracle, strand symmetry in canonical mode, a phage segment inside a bacterial
record found as a region, and the command line."""
import numpy as np
import pytest
import torch

from oracle import c_oracle
from oracle import phamers_oracle as po
from test_windows_cpu import window_table

pytestmark = pytest.mark.gpu
TOL = 1e-5
COMP = bytes.maketrans(b"ATGCN", b"TACGN")


def _device(blob, off):
    d = torch.zeros(((len(blob) + 15) // 16 * 16 + 16,), dtype=torch.uint8, device="cuda")
    if len(blob):
        d[:len(blob)] = torch.from_numpy(np.ascontiguousarray(blob)).cuda()
    return d[:len(blob)], torch.from_numpy(np.asarray(off, dtype=np.int64)).cuda()


def _records(seqs):
    blob = np.frombuffer(b"".join(seqs), dtype=np.uint8) if seqs else np.zeros(0, dtype=np.uint8)
    off = np.concatenate(([0], np.cumsum([len(s) for s in seqs]))).astype(np.int64)
    return blob, off


def _materialise(blob, off, window, step):
    """The windows as records of their own: (window blob, window offsets, spans, record of each window)."""
    wo, spans = window_table(np.diff(off), window, step)
    rec = np.repeat(np.arange(len(off) - 1), np.diff(wo))
    starts, ends = off[rec] + spans[:, 0], off[rec] + spans[:, 1]
    pieces = [blob[a:b] for a, b in zip(starts, ends)]
    wblob = np.concatenate(pieces) if pieces else np.zeros(0, dtype=np.uint8)
    woff = np.concatenate(([0], np.cumsum(ends - starts))).astype(np.int64)
    return wblob, woff, wo, spans, rec


def _random_bases(rng, n, gc=0.5):
    p = np.array([(1 - gc) / 2, (1 - gc) / 2, gc / 2, gc / 2])
    return rng.choice(np.frombuffer(b"ATGC", dtype=np.uint8), size=n, p=p)


def _edge_records(rng, window, step, k):
    """Records that put every edge case on some window: empty, shorter than k, aligned starts (the first records are 512-multiples
    long, so windows with steps of 16 / 256 bases start and end on 16- and 512-byte boundaries), unaligned starts, N and lower-case
    runs on window starts and ends."""
    lengths = [4096, 1024, 0, max(k - 1, 0), 1, window - 1, window, window + 1, window + step, window + 3 * step + 1, 4 * window + 7,
               2 * window + step // 2 + 5, 511, 512, 513, 9001]
    lengths += [int(x) for x in rng.integers(1, 6 * window + 20, size=6)]
    seqs = []
    for length in lengths:
        s = _random_bases(rng, length, float(rng.uniform(0.3, 0.7)))
        for edge in range(0, length, max(step, 1)):
            if rng.random() < 0.3:
                for pos in (edge, min(edge + window, length) - 1):                 # a window's first / last base
                    if 0 <= pos < length:
                        run = int(rng.integers(1, 4))
                        s[pos:pos + run] = ord("N") if rng.random() < 0.5 else rng.choice(np.frombuffer(b"atgcn", dtype=np.uint8))
        seqs.append(s.tobytes())
    return seqs


def _check_counts(blob, off, window, step, k, canonical, counts=True, freq=False):
    from phamers_b200 import ops
    d_seq, d_off = _device(blob, off)
    wblob, woff, want_wo, want_spans, _ = _materialise(blob, off, window, step)
    wo = ops.window_offsets_cuda(d_off, window, step)
    assert np.array_equal(wo.cpu().numpy(), want_wo)
    c, f, sp = ops.count_windows_cuda(d_seq, d_off, wo, window, step, k, canonical=canonical, counts=counts, freq=freq, spans=True)
    assert np.array_equal(sp.cpu().numpy(), want_spans)
    want = c_oracle.count(wblob, woff, k)
    if canonical:
        want = po.canonical_fold(want, k)
    if counts:
        assert np.array_equal(c.cpu().numpy().view(np.uint32).astype(np.int64), want), (window, step, k, canonical)
    if freq:
        d_wseq, d_woff = _device(wblob, woff)
        _, f_want = ops.count_cuda(d_wseq, d_woff, k, canonical=canonical, counts=False, freq=True)
        assert torch.equal(torch.nan_to_num(f, nan=-1.0), torch.nan_to_num(f_want, nan=-1.0)), (window, step, k, canonical)
    return wo, c, f, sp


@pytest.mark.parametrize("window,step", [(1000, 300), (512, 256), (160, 16), (37, 50), (3, 2)])
@pytest.mark.parametrize("canonical", [False, True])
def test_counts_bit_exact(window, step, canonical):
    rng = np.random.default_rng(window * 7 + step + canonical)
    blob, off = _records(_edge_records(rng, window, step, 6))
    for k in range(1, 7):
        _check_counts(blob, off, window, step, k, canonical)


@pytest.mark.parametrize("window,step", [(140000, 50000), (300000, 70001), (131072, 131072)])
def test_tiled_windows(window, step):
    """Windows of 131 072 bases and more are counted in tiles; records shorter than the window give shorter windows, tiled or not."""
    rng = np.random.default_rng(window + step)
    lengths = [400001, 100, 135000, 200000, 290017, 0, 5, 131071]
    seqs = []
    for length in lengths:
        s = _random_bases(rng, length, 0.6)
        for _ in range(length // 20000):
            a = int(rng.integers(0, length - 10))
            s[a:a + 10] = ord("N")
        seqs.append(s.tobytes())
    blob, off = _records(seqs)
    for k in (1, 4, 5, 6):
        for canonical in (False, True):
            _check_counts(blob, off, window, step, k, canonical, counts=True, freq=True)
    for k in (4, 5):
        _check_counts(blob, off, window, step, k, False, counts=False, freq=True)


def test_counts_features_and_both():
    rng = np.random.default_rng(11)
    blob, off = _records(_edge_records(rng, 700, 250, 6))
    for k in (2, 4, 5):
        for canonical in (False, True):
            _, c_only, f_none, _ = _check_counts(blob, off, 700, 250, k, canonical, counts=True, freq=False)
            _, c_none, f_only, _ = _check_counts(blob, off, 700, 250, k, canonical, counts=False, freq=True)
            _, c_both, f_both, _ = _check_counts(blob, off, 700, 250, k, canonical, counts=True, freq=True)
            assert f_none is None and c_none is None
            assert torch.equal(c_only, c_both) and torch.equal(torch.nan_to_num(f_only), torch.nan_to_num(f_both))


def test_slices_equal_one_call():
    from phamers_b200 import ops
    rng = np.random.default_rng(12)
    blob, off = _records(_edge_records(rng, 900, 200, 4) + [_random_bases(rng, 300000).tobytes()])
    d_seq, d_off = _device(blob, off)
    for window, step, canonical in ((900, 200, False), (900, 200, True), (140000, 30000, False)):
        wo = ops.window_offsets_cuda(d_off, window, step)
        total = int(wo[-1])
        whole_c, whole_f, whole_s = ops.count_windows_cuda(d_seq, d_off, wo, window, step, 4, canonical=canonical, freq=True, spans=True)
        for parts in range(2, 8):
            cuts = np.unique(np.concatenate(([0, total], rng.integers(0, total, size=parts - 1))))
            got = [ops.count_windows_cuda(d_seq, d_off, wo, window, step, 4, first=int(a), n=int(b - a), canonical=canonical, freq=True,
                                          spans=True) for a, b in zip(cuts[:-1], cuts[1:])]
            assert torch.equal(torch.cat([g[0] for g in got]), whole_c)
            assert torch.equal(torch.cat([g[2] for g in got]), whole_s)
            assert torch.equal(torch.nan_to_num(torch.cat([g[1] for g in got])), torch.nan_to_num(whole_f))
        with pytest.raises(Exception, match="outside"):
            ops.count_windows_cuda(d_seq, d_off, wo, window, step, 4, first=total - 1, n=2)


# ---------------------------------------------------------------------------------------------------------------------
# scores
# ---------------------------------------------------------------------------------------------------------------------
def _score_records(rng, n=60):
    seqs = []
    for _ in range(n):
        s = _random_bases(rng, int(rng.integers(2000, 30000)), float(rng.uniform(0.3, 0.7)))
        a = int(rng.integers(0, len(s) - 30))
        s[a:a + 30] = ord("N")
        seqs.append(s.tobytes())
    return _records(seqs)


@pytest.mark.parametrize("canonical", [False, True])
def test_window_scores(canonical):
    from phamers_b200 import ops, pipeline, references
    rng = np.random.default_rng(100 + canonical)
    blob, off = _score_records(rng)
    d_seq, d_off = _device(blob, off)
    scorer = pipeline.ContigScorer(canonical=canonical)
    wblob, woff, want_wo, want_spans, _ = _materialise(blob, off, 5000, 1000)
    for method, key in (("combo", 2), ("knn", 0), ("kmeans", 1)):
        wo, spans, scores = scorer.score_windows_device(d_seq, d_off, 5000, 1000, method=method)
        assert np.array_equal(wo.cpu().numpy(), want_wo) and np.array_equal(spans.cpu().numpy(), want_spans)
        # the same rows counted as records of their own and scored in one call: bit for bit
        d_wseq, d_woff = _device(wblob, woff)
        counts, _ = ops.count_cuda(d_wseq, d_woff, 4, canonical=canonical)
        want = ops.score_cuda(counts, scorer.refs, scorer.n_positive, scorer.cent_pos, scorer.cent_neg, scorer.k_neighbors)[key]
        assert torch.equal(scores, want), method
    # other slice sizes: the exhaustive roads may sum in another order
    _, _, combo = scorer.score_windows_device(d_seq, d_off, 5000, 1000)
    for slice_ in (97, 1000):
        scorer.WINDOW_SLICE = slice_
        _, _, other = scorer.score_windows_device(d_seq, d_off, 5000, 1000)
        assert torch.max(torch.abs(other - combo)).item() <= 1e-12 and torch.equal(torch.sign(other), torch.sign(combo)), slice_
    del scorer.WINDOW_SLICE
    # the oracle
    X = c_oracle.count(wblob, woff, 4)
    X = po.normalize_counts(po.canonical_fold(X, 4) if canonical else X)
    pos, neg = references.load_reference_features(equalize=True, canonical=canonical)
    want = po.score_points(X, pos, neg, centroids=references.reference_centroids(pos, neg))
    got = combo.cpu().numpy()
    assert np.max(np.abs(got - want)) <= TOL and np.array_equal(np.sign(got), np.sign(want))


def test_window_scores_from_features():
    """k_neighbors outside {1, 3, 5}: the windows are normalised on the device and scored as float64 feature rows."""
    from phamers_b200 import ops, pipeline
    rng = np.random.default_rng(7)
    blob, off = _score_records(rng, 30)
    d_seq, d_off = _device(blob, off)
    scorer = pipeline.ContigScorer(k_neighbors=7)
    _, _, scores = scorer.score_windows_device(d_seq, d_off, 4000, 1500)
    wblob, woff, _, _, _ = _materialise(blob, off, 4000, 1500)
    d_wseq, d_woff = _device(wblob, woff)
    _, feats = ops.count_cuda(d_wseq, d_woff, 4, counts=False, freq=True)
    want = ops.score_cuda(feats, scorer.refs, scorer.n_positive, scorer.cent_pos, scorer.cent_neg, 7)[2]
    assert torch.equal(scores, want)


def test_reverse_complement_windows_mirror():
    from phamers_b200 import ops, pipeline
    rng = np.random.default_rng(31)
    window, step = 5000, 1000
    seqs = []
    for length in (5000 + 1000 * 17, 5000 + 1000 * 40, 3000):                 # (L - w) % s == 0: the windows mirror
        s = _random_bases(rng, length, 0.45)
        s[100:120] = ord("N")
        fwd = s.tobytes()
        seqs += [fwd, fwd.translate(COMP)[::-1]]
    blob, off = _records(seqs)
    d_seq, d_off = _device(blob, off)
    scorer = pipeline.ContigScorer(canonical=True)
    wo, spans, scores = scorer.score_windows_device(d_seq, d_off, window, step)
    counts, _, _ = ops.count_windows_cuda(d_seq, d_off, wo, window, step, 4, canonical=True)
    wo = wo.cpu().numpy()
    for r in range(0, len(seqs), 2):
        a, b = slice(wo[r], wo[r + 1]), slice(wo[r + 1], wo[r + 2])
        assert torch.equal(scores[a], scores[b].flip(0)) and torch.equal(counts[a], counts[b].flip(0)), r
        length = off[r + 1] - off[r]
        sp = spans.cpu().numpy()
        assert np.array_equal(sp[a], length - sp[b][::-1, ::-1]), r


# ---------------------------------------------------------------------------------------------------------------------
# the point of the feature: a phage segment inside a bacterial record
# ---------------------------------------------------------------------------------------------------------------------
def _chain(row):
    """3rd-order Markov chain of a 4-mer count row: P(next base | previous three bases), cumulative."""
    t = row.reshape(64, 4).astype(np.float64) + 0.5
    return np.cumsum(t / t.sum(axis=1, keepdims=True), axis=1)


def _generate(cum, n, rng):
    u = rng.random(n)
    out = np.empty(n, dtype=np.uint8)
    sym = np.frombuffer(b"ATGC", dtype=np.uint8)
    state = 0
    for i in range(n):
        b = min(int(np.searchsorted(cum[state], u[i], side="right")), 3)
        out[i] = sym[b]
        state = ((state << 2) | b) & 63
    return out


def test_prophage_found_as_region():
    from phamers_b200 import pipeline, references
    _, pos_c, _, neg_c = references.load_reference_counts()
    rng = np.random.default_rng(2026)
    seqs, inserts = [], []
    for bac, phage, size in ((1144, 615, 40000), (1237, 1866, 30000), (1825, 579, 50000)):
        left, right = int(rng.integers(100000, 160000)), int(rng.integers(100000, 160000))
        parts = (_generate(_chain(neg_c[bac]), left, rng), _generate(_chain(pos_c[phage]), size, rng),
                 _generate(_chain(neg_c[bac]), right, rng))
        seqs.append(np.concatenate(parts).tobytes())
        inserts.append((left, left + size))
    blob, off = _records(seqs)
    d_seq, d_off = _device(blob, off)
    scorer = pipeline.ContigScorer()
    _, whole = scorer.score_device(d_seq, d_off)
    assert (whole.cpu().numpy() < 0).all()                              # one score per record hides the phage
    from phamers_b200 import phamer
    wo, spans, scores = scorer.score_windows_device(d_seq, d_off, 5000, 1000)
    sc = phamer.phamer_scorer()
    sc.window_records = np.repeat(np.arange(len(seqs)), np.diff(wo.cpu().numpy()))
    sc.window_ids = sc.window_records.astype(str)
    sc.window_spans, sc.window_scores = spans.cpu().numpy(), scores.cpu().numpy()
    sc.find_regions()
    for r, (a, b) in enumerate(inserts):
        mine = sc.region_ids == str(r)
        assert mine.any(), r
        rs = sc.region_spans[mine]
        covered = np.minimum(rs[:, 1], b) - np.maximum(rs[:, 0], a)
        assert covered.max() >= 0.8 * (b - a), (r, rs, (a, b))
        assert ((rs[:, 1] > a - 5000) & (rs[:, 0] < b + 5000)).all(), (r, rs, (a, b))       # no region far from the segment


# ---------------------------------------------------------------------------------------------------------------------
# command line
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("canonical", [False, True])
def test_cli_windows(tmp_path, canonical):
    from phamers_b200 import fileIO, phamer, references
    from test_gpu_cli import _write_fasta
    rng = np.random.default_rng(5000 + canonical)
    indir = tmp_path / "sample"
    indir.mkdir()
    lengths, seqs = _write_fasta(indir / "contigs.fasta", rng, 80)
    flags = ["-canonical"] if canonical else []
    out = tmp_path / "out"
    phamer.main(["-in", str(indir), "-out", str(out), "-equal"] + flags)
    plain = open(out / "phamer_scores.csv", "rb").read()
    scorer = phamer.main(["-in", str(indir), "-out", str(out), "-window", "5000", "-step", "1000", "-equal"] + flags)
    assert open(out / "phamer_scores.csv", "rb").read() == plain
    ids, spans, got = fileIO.read_phamer_windows(str(out / "phamer_windows.csv"))
    blob, off = _records([s.encode() for s in seqs])
    keep = lengths >= 5000
    wblob, woff, wo, want_spans, rec = _materialise(blob, off, 5000, 1000)
    in_kept = keep[rec]
    assert ids.tolist() == [str(r) for r in rec[in_kept]]
    assert np.array_equal(spans, want_spans[in_kept])
    assert np.array_equal(got, scorer.window_scores)
    X = c_oracle.count(wblob, woff, 4)[in_kept]
    X = po.normalize_counts(po.canonical_fold(X, 4) if canonical else X)
    pos, neg = references.load_reference_features(equalize=True, canonical=canonical)
    want = po.score_points(X, pos, neg, centroids=references.reference_centroids(pos, neg))
    assert np.max(np.abs(got - want)) <= TOL and np.array_equal(np.sign(got), np.sign(want))
    r_ids, r_spans, r_windows, r_mean, r_max = fileIO.read_phamer_regions(str(out / "phamer_regions.csv"))
    assert r_windows.sum() == (got >= 0).sum() and (r_max >= 0).all() and (r_mean <= r_max).all()
    assert set(r_ids) <= set(ids)

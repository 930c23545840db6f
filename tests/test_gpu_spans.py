"""GPU checks of span scoring: span counts bit for bit against the C oracle on the span slices materialised as records (plain and
canonical, k = 1..6; unsorted, overlapping, duplicated, empty and shorter-than-k spans, every start offset mod 16, 512-byte boundaries,
N / lower-case runs at the edges, tiled spans at and around SPLIT_MIN, whole records), spans equal to the records and to the windows,
invalid spans and list overflow, scores and neighbour reports against the same bases scored as records of their own, strand symmetry,
slicing, and the command line."""

import numpy as np
import pytest
import torch

from oracle import c_oracle
from oracle import phamers_oracle as po
from test_gpu_windows import _chain, _device, _generate, _random_bases, _records

pytestmark = pytest.mark.gpu
SPLIT_MIN = 131072
COMP = bytes.maketrans(b"ATGCN", b"TACGN")


def _materialise(blob, off, spans):
    """The spans as records of their own: (blob, offsets)."""
    pieces = [blob[off[r] + a:off[r] + b] for r, a, b in spans]
    sblob = np.concatenate(pieces) if pieces else np.zeros(0, dtype=np.uint8)
    soff = np.concatenate(([0], np.cumsum([b - a for _, a, b in spans]))).astype(np.int64)
    return sblob, soff


def _edge_case_records(rng):
    """Records with N and lower-case runs at known places: (records, [(record, position)] of the runs)."""
    lengths = [0, 3, 1000, 5000, 20011, 4096, SPLIT_MIN + 3000, 400001]
    seqs, runs = [], []
    for r, length in enumerate(lengths):
        s = _random_bases(rng, length, float(rng.uniform(0.3, 0.7)))
        for _ in range(length // 3000):
            pos = int(rng.integers(0, length - 4))
            width = int(rng.integers(1, 4))
            s[pos:pos + width] = ord("N") if rng.random() < 0.5 else rng.choice(np.frombuffer(b"atgcn", dtype=np.uint8))
            runs.append((r, pos, width))
        seqs.append(s.tobytes())
    return seqs, runs


def _edge_case_spans(rng, lengths, runs, k=6):
    L = list(lengths)
    spans = []
    for r, length in enumerate(L):
        spans.append((r, 0, length))                                              # whole record
        spans.append((r, length, length))                                         # empty, at the end
    nonempty = [r for r, n in enumerate(L) if n >= 600]
    for _ in range(60):                                                           # random, unsorted, overlapping
        r = int(rng.choice(nonempty))
        a, b = np.sort(rng.integers(0, L[r] + 1, size=2))
        spans.append((r, int(a), int(b)))
    for j in range(16):                                                           # every start offset mod 16, 512-byte boundaries
        r = nonempty[j % len(nonempty)]
        m = int(rng.integers(1, max(2, L[r] // 512)))
        a = min(512 * m - 16 + j, L[r] - 1)
        spans.append((r, a, min(L[r], a + 512 + int(rng.integers(0, 40)))))
        spans.append((r, 16 * int(rng.integers(0, L[r] // 16)) + j, 0))
        spans[-1] = (spans[-1][0], min(spans[-1][1], L[r]), min(L[r], spans[-1][1] + int(rng.integers(0, 700))))
    for length in range(0, k + 1):                                                # empty and shorter than k
        r = nonempty[length % len(nonempty)]
        a = int(rng.integers(0, L[r] - length))
        spans.append((r, a, a + length))
    for r, pos, width in runs[:40]:                                               # runs at the first / last bases of a span
        spans.append((r, pos, min(L[r], pos + 300)))
        spans.append((r, max(0, pos + width - 300), pos + width))
        spans.append((r, max(0, pos - 2), min(L[r], pos + width + 2)))
    big = [r for r, n in enumerate(L) if n >= SPLIT_MIN + 2]
    for r in big:                                                                 # tiled spans: at SPLIT_MIN and either side
        for length in (SPLIT_MIN - 1, SPLIT_MIN, SPLIT_MIN + 1, L[r] - 5):
            a = int(rng.integers(0, L[r] - length + 1))
            spans.append((r, a, a + length))
    spans += [spans[i] for i in rng.integers(0, len(spans), size=10)]             # duplicates
    order = rng.permutation(len(spans))
    return np.array([spans[i] for i in order], dtype=np.int64).reshape(-1, 3)


def _check_counts(blob, off, spans, k, canonical, counts=True, freq=False):
    from phamers_b200 import ops
    d_seq, d_off = _device(blob, off)
    c, f = ops.count_spans_cuda(d_seq, d_off, torch.from_numpy(spans).cuda(), k, canonical=canonical, counts=counts, freq=freq)
    sblob, soff = _materialise(blob, off, spans)
    if counts:
        want = c_oracle.count(sblob, soff, k)
        if canonical:
            want = po.canonical_fold(want, k)
        assert np.array_equal(c.cpu().numpy().view(np.uint32).astype(np.int64), want), (k, canonical)
    if freq:
        d_sseq, d_soff = _device(sblob, soff)
        _, f_want = ops.count_cuda(d_sseq, d_soff, k, canonical=canonical, counts=False, freq=True)
        assert torch.equal(torch.nan_to_num(f, nan=-1.0), torch.nan_to_num(f_want, nan=-1.0)), (k, canonical)
    return c, f


@pytest.mark.parametrize("canonical", [False, True])
def test_counts_bit_exact(canonical):
    rng = np.random.default_rng(40 + canonical)
    seqs, runs = _edge_case_records(rng)
    blob, off = _records(seqs)
    spans = _edge_case_spans(rng, np.diff(off), runs)
    assert (spans[:, 2] - spans[:, 1] >= SPLIT_MIN).sum() >= 6 and (spans[:, 2] == spans[:, 1]).sum() >= 8
    for k in range(1, 7):
        _check_counts(blob, off, spans, k, canonical)


def test_counts_features_and_both():
    rng = np.random.default_rng(41)
    seqs, runs = _edge_case_records(rng)
    blob, off = _records(seqs)
    spans = _edge_case_spans(rng, np.diff(off), runs)
    for k in (2, 4, 5, 6):
        for canonical in (False, True):
            c_only, f_none = _check_counts(blob, off, spans, k, canonical, counts=True, freq=False)
            c_none, f_only = _check_counts(blob, off, spans, k, canonical, counts=False, freq=True)
            c_both, f_both = _check_counts(blob, off, spans, k, canonical, counts=True, freq=True)
            assert f_none is None and c_none is None
            assert torch.equal(c_only, c_both) and torch.equal(torch.nan_to_num(f_only), torch.nan_to_num(f_both))


def test_spans_equal_records_and_windows():
    from phamers_b200 import ops
    rng = np.random.default_rng(42)
    seqs, _ = _edge_case_records(rng)
    blob, off = _records(seqs)
    d_seq, d_off = _device(blob, off)
    n = len(seqs)
    lengths = np.diff(off)
    whole = torch.from_numpy(np.stack((np.arange(n), np.zeros(n, dtype=np.int64), lengths), axis=1)).cuda()
    for k in (1, 4, 5, 6):
        for canonical in (False, True):
            c, f = ops.count_spans_cuda(d_seq, d_off, whole, k, canonical=canonical, freq=True)
            c_want, f_want = ops.count_cuda(d_seq, d_off, k, canonical=canonical, freq=True)
            assert torch.equal(c, c_want) and torch.equal(torch.nan_to_num(f), torch.nan_to_num(f_want)), (k, canonical)
    for window, step in ((5000, 1000), (140000, 60000)):
        wo = ops.window_offsets_cuda(d_off, window, step)
        c_want, f_want, sp = ops.count_windows_cuda(d_seq, d_off, wo, window, step, 4, freq=True, spans=True)
        rec = torch.repeat_interleave(torch.arange(n, device="cuda"), torch.diff(wo))
        c, f = ops.count_spans_cuda(d_seq, d_off, torch.cat((rec[:, None], sp), dim=1).contiguous(), 4, freq=True)
        assert torch.equal(c, c_want) and torch.equal(torch.nan_to_num(f), torch.nan_to_num(f_want)), window


def test_invalid_spans_and_list_overflow():
    from phamers_b200 import _lib, ops
    lib = _lib.load()
    rng = np.random.default_rng(43)
    seqs = [_random_bases(rng, n).tobytes() for n in (1000, 300000, 50)]
    blob, off = _records(seqs)
    d_seq, d_off = _device(blob, off)
    good = [(0, 0, 1000), (1, 5, 299000), (2, 10, 20), (0, 1000, 1000)]
    bads = [((3, 0, 1), "names no record"), ((-1, 0, 1), "names no record"), ((0, -1, 5), "starts before"),
            ((2, 30, 29), "ends before it starts"), ((2, 0, 51), "ends past its record"), ((1, 299999, 300001), "ends past")]
    for bad, msg in bads:
        for at in (1, 3):
            table = good[:at] + [bad] + good[at:] + [(3, 0, 0), (0, 5, 1)]        # a later invalid span is not the one named
            spans = torch.tensor(table, dtype=torch.int64, device="cuda")
            n = len(table)
            counts = torch.full((n, 256), 7, dtype=torch.int32, device="cuda")
            freq = torch.full((n, 256), 0.5, dtype=torch.float64, device="cuda")
            ws = torch.empty((lib.phm_kmer_count_spans_workspace_bytes(n, 1 << 20, 4, 0),), dtype=torch.uint8, device="cuda")
            rc = lib.phm_kmer_count_spans(_lib.ptr(d_seq), _lib.ptr(d_off), 3, _lib.ptr(spans), n, 4, 0, _lib.ptr(counts),
                                          _lib.ptr(freq), _lib.ptr(ws), ws.numel(), _lib.stream_ptr())
            err = lib.phm_last_error().decode()
            assert rc == -1 and ("span %d " % at) in err and msg in err, (bad, at, err)
            assert (counts == 7).all() and (freq == 0.5).all(), bad                # no output row written
            with pytest.raises(_lib.PhamersLibraryError, match="span %d " % at):
                ops.count_spans_cuda(d_seq, d_off, spans, 4)
    # the exact list does not fit: one item per span, but the 300 000-base span needs 4 tiles
    spans = torch.tensor(good, dtype=torch.int64, device="cuda")
    counts = torch.full((4, 256), 7, dtype=torch.int32, device="cuda")
    fixed = lib.phm_kmer_count_spans_workspace_bytes(0, 0, 4, 0)
    ws = torch.empty((fixed + 4 * 32,), dtype=torch.uint8, device="cuda")          # exactly four items: the list needs seven
    rc = lib.phm_kmer_count_spans(_lib.ptr(d_seq), _lib.ptr(d_off), 3, _lib.ptr(spans), 4, 4, 0, _lib.ptr(counts), None,
                                  _lib.ptr(ws), ws.numel(), _lib.stream_ptr())
    assert rc == -3 and b"workspace too small" in lib.phm_last_error() and (counts == 7).all()
    c, _ = ops.count_spans_cuda(d_seq, d_off, spans, 4)                          # sized from the span lengths: fits
    sblob, soff = _materialise(blob, off, np.array(good))
    assert np.array_equal(c.cpu().numpy().astype(np.int64), c_oracle.count(sblob, soff, 4))


# ---------------------------------------------------------------------------------------------------------------------
# scores and neighbour reports: the standalone-record oracle
# ---------------------------------------------------------------------------------------------------------------------
def _write_fasta(path, seqs, names):
    with open(path, "w") as fh:
        for name, s in zip(names, seqs):
            fh.write(">%s some description\n%s\n" % (name, s.decode("latin-1")))


def _score_case(rng):
    seqs = []
    for _ in range(40):
        s = _random_bases(rng, int(rng.integers(3000, 40000)), float(rng.uniform(0.3, 0.7)))
        a = int(rng.integers(0, len(s) - 110))
        s[a:a + 30] = ord("N")
        s[a + 100:a + 110] = np.frombuffer(b"acgtnacgta", dtype=np.uint8)
        seqs.append(s.tobytes())
    lengths = [len(s) for s in seqs]
    spans = []
    for _ in range(300):
        r = int(rng.integers(0, len(seqs)))
        a = int(rng.integers(0, lengths[r]))
        spans.append((r, a, min(lengths[r], a + int(rng.integers(1, 20000)))))
    spans += [(0, 10, 10), (1, 5, 7), (2, 0, lengths[2])]                         # no k-mer, one short of k, a whole record
    spans += spans[:5]
    return seqs, np.array(spans, dtype=np.int64)


@pytest.mark.parametrize("canonical", [False, True])
@pytest.mark.parametrize("k_neighbors", [3, 7])
def test_scores_and_neighbors_equal_standalone_records(tmp_path, canonical, k_neighbors):
    from phamers_b200 import fileIO, ops, phamer, pipeline
    rng = np.random.default_rng(50 + canonical + 2 * k_neighbors)
    seqs, spans = _score_case(rng)
    blob, off = _records(seqs)
    names = ["CTG%d.1" % i for i in range(len(seqs))]                             # GenBank-style: these are the score-file ids
    contigs = tmp_path / "contigs.fasta"
    _write_fasta(contigs, seqs, names)
    sblob, soff = _materialise(blob, off, spans)
    pieces = [sblob[soff[i]:soff[i + 1]].tobytes() for i in range(len(spans))]
    alone = tmp_path / "alone.fasta"
    _write_fasta(alone, pieces, ["S%d.1" % i for i in range(len(spans))])
    d_seq, d_off = _device(blob, off)
    d_spans = torch.from_numpy(spans).cuda()
    scorer = pipeline.ContigScorer(k_neighbors=k_neighbors, canonical=canonical)

    def standalone(method):
        if k_neighbors in (1, 3, 5):
            return scorer.score_fasta(str(alone), method=method)[1]
        # score_fasta takes the count road only; other shapes score the records' feature rows
        _, a_seq, a_off = fileIO.read_fasta_arrays_cuda(str(alone))
        _, feats = ops.count_cuda(a_seq, a_off, 4, canonical=canonical, counts=False, freq=True)
        out = ops.score_cuda(feats, scorer.refs, scorer.n_positive, scorer.cent_pos, scorer.cent_neg, k_neighbors)
        return out[{"knn": 0, "kmeans": 1, "combo": 2}[method]].cpu().numpy()

    for method in ("combo", "knn", "kmeans"):
        got = scorer.score_spans_device(d_seq, d_off, d_spans, method=method)
        want = standalone(method)
        assert np.array_equal(got.cpu().numpy(), want, equal_nan=True), method
        host = scorer.score_spans_fasta(str(contigs), np.array(names)[spans[:, 0]], spans[:, 1:], method=method)
        assert np.array_equal(host, want, equal_nan=True), method
    assert np.isnan(want[-8]) and np.isnan(want[-7]) and not np.isnan(want[-6])
    # neighbour reports: phamer_scorer.score_neighbors on the spans written as records, score_spans on the contigs
    for method in ("combo", "knn"):
        ref = phamer.phamer_scorer()
        ref.fasta_file, ref.canonical, ref.k_neighbors, ref.scoring_method = str(alone), canonical, k_neighbors, method
        ref.load_reference_data()
        ref.load_data(length_requirement=0)
        want = ref.score_neighbors()
        sc = phamer.phamer_scorer()
        sc.fasta_file, sc.canonical, sc.k_neighbors, sc.scoring_method = str(contigs), canonical, k_neighbors, method
        sc.load_reference_data()
        got = sc.score_spans(np.array(names)[spans[:, 0]], spans[:, 1:])
        assert np.array_equal(got, want, equal_nan=True), method
        assert np.array_equal(sc.span_neighbor_ids, ref.neighbor_ids) and np.array_equal(sc.span_neighbor_labels, ref.neighbor_labels)
        assert np.array_equal(sc.span_neighbor_distances, ref.neighbor_distances, equal_nan=True)
        assert np.array_equal(sc.span_nearest_clusters, ref.nearest_clusters)
        assert np.array_equal(sc.span_nearest_cluster_distances, ref.nearest_cluster_distances, equal_nan=True)
        assert (sc.span_neighbor_labels[-8] == -1).all() and (sc.span_nearest_clusters[-8] == -1).all()
    # names by first token when no score-file id matches; bad coordinates name their source line
    tokens = ["ctg_%d" % i for i in range(len(seqs))]
    _write_fasta(contigs, seqs, tokens)
    host = scorer.score_spans_fasta(str(contigs), np.array(tokens)[spans[:, 0]], spans[:, 1:])
    assert np.array_equal(host, standalone("combo"), equal_nan=True)
    with pytest.raises(ValueError, match="x.bed line 9"):
        scorer.score_spans_fasta(str(contigs), ["ctg_0"], [[0, len(seqs[0]) + 1]], lines=["x.bed line 9"])


def test_reverse_complement_span_mirrors():
    from phamers_b200 import pipeline
    rng = np.random.default_rng(44)
    seqs = []
    for length in (30000, 9000, 200000):
        s = _random_bases(rng, length, 0.45)
        s[100:120] = ord("N")
        fwd = s.tobytes()
        seqs += [fwd, fwd.translate(COMP)[::-1]]
    blob, off = _records(seqs)
    d_seq, d_off = _device(blob, off)
    table = []
    for r in range(0, len(seqs), 2):
        length = len(seqs[r])
        for _ in range(20):
            a, b = np.sort(rng.integers(0, length + 1, size=2))
            table += [(r, int(a), int(b)), (r + 1, length - int(b), length - int(a))]
    table.append((4, 1000, 1000 + SPLIT_MIN + 7))
    table.append((5, len(seqs[4]) - 1000 - SPLIT_MIN - 7, len(seqs[4]) - 1000))
    scorer = pipeline.ContigScorer(canonical=True)
    scores, ref_i, ref_d, cen_i, cen_d = scorer.score_spans_device(d_seq, d_off, torch.tensor(table, device="cuda"), neighbors=True)
    for out in (scores, ref_i, ref_d, cen_i, cen_d):
        assert torch.equal(torch.nan_to_num(out[0::2].double()), torch.nan_to_num(out[1::2].double()))


def test_slices_equal_one_call():
    from phamers_b200 import pipeline
    rng = np.random.default_rng(45)
    seqs, spans = _score_case(rng)
    blob, off = _records(seqs)
    d_seq, d_off = _device(blob, off)
    d_spans = torch.from_numpy(spans).cuda()
    for k_neighbors in (3, 7):
        scorer = pipeline.ContigScorer(k_neighbors=k_neighbors)
        whole = scorer.score_spans_device(d_seq, d_off, d_spans, neighbors=True)
        for slice_ in (1, 97, 250):
            scorer.SPAN_SLICE = slice_
            part = scorer.score_spans_device(d_seq, d_off, d_spans, neighbors=True)
            for a, b in zip(part, whole):
                assert torch.equal(torch.nan_to_num(a.double()), torch.nan_to_num(b.double())), (k_neighbors, slice_)
        assert scorer.score_spans_device(d_seq, d_off, d_spans[:0]).shape == (0,)


# ---------------------------------------------------------------------------------------------------------------------
# command line: a phage segment inside a bacterial record, found as a region and scored as one sequence
# ---------------------------------------------------------------------------------------------------------------------
def test_cli_region_scores_and_spans(tmp_path):
    from phamers_b200 import fileIO, phamer, references
    _, pos_c, _, neg_c = references.load_reference_counts()
    rng = np.random.default_rng(2026)
    left, size, right = 90000, 40000, 80000
    host = np.concatenate((_generate(_chain(neg_c[1144]), left, rng), _generate(_chain(pos_c[615]), size, rng),
                           _generate(_chain(neg_c[1144]), right, rng))).tobytes()
    other = _random_bases(rng, 30000).tobytes()
    indir = tmp_path / "sample"
    indir.mkdir()
    _write_fasta(indir / "contigs.fasta", [other, host], ["OTH1.1", "HOST1.1"])
    out = tmp_path / "out"
    base = ["-in", str(indir), "-out", str(out), "-neighbors", "-window", "5000", "-step", "1000"]
    phamer.main(base)
    names = ("phamer_scores.csv", "phamer_neighbors.csv", "phamer_windows.csv", "phamer_regions.csv")
    before = {n: open(out / n, "rb").read() for n in names}
    r_ids, r_spans = fileIO.read_phamer_regions(str(out / "phamer_regions.csv"))[:2]
    mine = np.flatnonzero(r_ids == "HOST1.1")
    assert len(mine), r_spans
    covered = np.minimum(r_spans[mine, 1], left + size) - np.maximum(r_spans[mine, 0], left)
    best = mine[int(np.argmax(covered))]
    assert covered.max() >= 0.8 * size
    bed = tmp_path / "regions.bed"
    bed.write_text("# the regions again, by first token\n" + "".join("%s\t%d\t%d\tr%d\n" % (i, a, b, j)
                                                                       for j, (i, (a, b)) in enumerate(zip(r_ids, r_spans))))
    scorer = phamer.main(base + ["-region_scores", "-spans", str(bed)])
    for n in names:
        assert open(out / n, "rb").read() == before[n], n
    rs = fileIO.read_phamer_spans(str(out / "phamer_region_scores.csv"))
    sp = fileIO.read_phamer_spans(str(out / "phamer_spans.csv"))
    assert np.array_equal(rs[0], r_ids) and np.array_equal(rs[1], r_spans) and (rs[2] == ".").all()
    assert np.array_equal(sp[0], r_ids) and np.array_equal(sp[1], r_spans) and sp[2].tolist() == ["r%d" % j for j in range(len(r_ids))]
    for a, b in zip(rs[3:], sp[3:]):
        assert np.array_equal(a, b)
    assert rs[3][best] >= 0                                                      # the region is phage-like on its own
    # the region's bases as a record of their own, scored the way the command line scores contigs
    a, b = r_spans[best]
    alone = tmp_path / "alone"
    alone.mkdir()
    _write_fasta(alone / "region.fasta", [host[a:b]], ["REG1.1"])
    ref = phamer.main(["-in", str(alone), "-out", str(tmp_path / "alone_out"), "-neighbors", "-l", "0"])
    assert rs[3][best] == ref.scores[0]
    assert rs[4][best].tolist() == ref.neighbor_ids[0].tolist() and rs[6][best].tolist() == ref.neighbor_distances[0].tolist()
    assert rs[7][best].tolist() == ref.nearest_clusters[0].tolist()
    assert np.array_equal(scorer.span_scores, sp[3])

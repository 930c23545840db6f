"""CPU-only checks of span scoring: the BED reader, the contig-name matching rules, the span file's round trip, the argument errors of
the span entry points (reported before a device is touched), and the command line's checks and file plumbing."""
import ctypes

import numpy as np
import pytest

import __graft_entry__ as entry


@pytest.fixture(scope="module")
def lib():
    entry.build()
    from phamers_b200 import _lib
    return _lib


# ---------------------------------------------------------------------------------------------------------------------
# BED
# ---------------------------------------------------------------------------------------------------------------------
def test_read_bed(tmp_path):
    from phamers_b200 import fileIO
    path = tmp_path / "a.bed"
    path.write_text("# a comment\n"
                    "track name=prophages\n"
                    "browser position chr1:1-100\n"
                    "\n"
                    "c1\t0\t100\tphage_1\t0\t+\textra\n"
                    "c2 5 5\n"
                    "   c1   7    9   gene  \n"
                    "NODE_1_length_50\t10\t40\n"
                    "\t\n")
    ids, spans, names = fileIO.read_bed(str(path))
    assert ids.tolist() == ["c1", "c2", "c1", "NODE_1_length_50"]
    assert spans.dtype == np.int64 and spans.tolist() == [[0, 100], [5, 5], [7, 9], [10, 40]]
    assert names.tolist() == ["phage_1", ".", "gene", "."]
    ids, spans, names, lines = fileIO.read_bed(str(path), with_lines=True)
    assert lines == ["%s line %d" % (path, n) for n in (5, 6, 7, 8)]
    empty = tmp_path / "e.bed"
    empty.write_text("# nothing\n")
    ids, spans, names = fileIO.read_bed(str(empty))
    assert len(ids) == 0 and spans.shape == (0, 2) and len(names) == 0


@pytest.mark.parametrize("line,msg", [("c1\t5\n", "chrom, start and end"), ("c1 x 7\n", "integers"), ("c1 5 7.5\n", "integers"),
                                      ("c1 -1 7\n", "not an interval"), ("c1 9 7\n", "not an interval")])
def test_read_bed_malformed(tmp_path, line, msg):
    from phamers_b200 import fileIO
    path = tmp_path / "bad.bed"
    path.write_text("# header\nc0\t0\t10\n" + line)
    with pytest.raises(ValueError, match="line 3: .*" + msg):
        fileIO.read_bed(str(path))


# ---------------------------------------------------------------------------------------------------------------------
# contig names -> records
# ---------------------------------------------------------------------------------------------------------------------
def test_match_records():
    from phamers_b200 import fileIO, pipeline
    tokens = ["NC_001416.1", "contig_ID_17", "plain", "dup", "dup", "AB000001.1", "other"]
    ids = [fileIO.get_id(t) for t in tokens]
    assert ids == ["NC_001416.1", "17", None, None, None, "AB000001.1", None]
    got = pipeline.match_records(["17", "NC_001416.1", "plain", "contig_ID_17", "other", "17"], ids, tokens)
    assert got.dtype == np.int64 and got.tolist() == [1, 0, 2, 1, 6, 1]
    # a score-file id wins over a first token that happens to be the same text
    assert pipeline.match_records(["x"], ["x", None], ["y", "x"]).tolist() == [0]
    with pytest.raises(ValueError, match="'dup' names 2 records"):
        pipeline.match_records(["plain", "dup"], ids, tokens)
    with pytest.raises(ValueError, match="'missing' names no record"):
        pipeline.match_records(["missing"], ids, tokens)
    with pytest.raises(ValueError, match="'a' names 2 records"):
        pipeline.match_records(["a"], ["a", "a"], ["r0", "r1"])
    assert pipeline.match_records([], ids, tokens).shape == (0,)


# ---------------------------------------------------------------------------------------------------------------------
# span file
# ---------------------------------------------------------------------------------------------------------------------
def test_span_file_round_trip(tmp_path):
    from phamers_b200 import fileIO
    rng = np.random.default_rng(9)
    n, k = 150, 3
    ids = np.array(["c%d" % i for i in rng.integers(0, 40, size=n)])
    spans = np.sort(rng.integers(0, 1 << 40, size=(n, 2)), axis=1)
    names = np.array(["g%d" % i if i % 3 else "." for i in range(n)])
    scores = rng.normal(size=n) * 10.0 ** rng.integers(-20, 3, size=n)
    refs = np.array([["NC_%06d.1" % v for v in row] for row in rng.integers(0, 999999, size=(n, k))])
    labels = rng.integers(0, 2, size=(n, k))
    dist = rng.random((n, k)) * 10.0 ** rng.integers(-17, 0, size=(n, k))
    clusters = rng.integers(-1, 86, size=(n, 2))
    cdist = rng.random((n, 2))
    scores[4] = np.nan                                                   # a span without a countable k-mer
    refs[4], labels[4], dist[4], clusters[4], cdist[4] = "", -1, np.nan, -1, np.nan
    path = str(tmp_path / "s.csv")
    fileIO.save_phamer_spans(ids, spans, names, scores, refs, labels, dist, clusters, cdist, path)
    back = fileIO.read_phamer_spans(path)
    for a, b in zip(back, (ids, spans, names, scores, refs, labels, dist, clusters, cdist)):
        assert np.array_equal(a, b, equal_nan=a.dtype.kind == "f")
    text = open(path).read().splitlines()
    assert text[0] == "# PhaMers span file"
    assert text[1] == ("# id, start, end, name, score, reference_1, class_1, distance_1, reference_2, class_2, distance_2, reference_3, "
                       "class_3, distance_3, phage_cluster, phage_cluster_distance, bacteria_cluster, bacteria_cluster_distance")
    fileIO.save_phamer_spans([], np.zeros((0, 2)), [], [], np.zeros((0, k), dtype=str), np.zeros((0, k)), np.zeros((0, k)),
                             np.zeros((0, 2)), np.zeros((0, 2)), path)
    assert [len(a) for a in fileIO.read_phamer_spans(path)] == [0] * 9


# ---------------------------------------------------------------------------------------------------------------------
# argument errors of the entry points: reported through phm_last_error before any device is touched
# ---------------------------------------------------------------------------------------------------------------------
def test_span_symbols_load(lib):
    handle = lib.load()
    for name in ("phm_kmer_count_spans_workspace_bytes", "phm_kmer_count_spans"):
        assert getattr(handle, name).argtypes == lib.SIGNATURES[name][1]
    fixed = handle.phm_kmer_count_spans_workspace_bytes(0, 0, 4, 0)
    assert fixed % 256 == 0
    assert handle.phm_kmer_count_spans_workspace_bytes(1000, 5000, 4, 0) == fixed + 32000
    assert handle.phm_kmer_count_spans_workspace_bytes(1000, 10 * 65536 + 5, 4, 0) == fixed + 32512      # 1010 items, 256-byte granules
    assert handle.phm_kmer_count_spans_workspace_bytes(-5, -7, 4, 0) == fixed


def test_count_spans_argument_errors(lib):
    handle = lib.load()
    seq, off, spans, counts, ws = (ctypes.c_void_p(v) for v in (1 << 20, 2 << 20, 3 << 20, 4 << 20, 5 << 20))
    big = 1 << 30

    def call(seq=seq, off=off, n_rec=10, spans=spans, n=5, k=4, flags=0, counts=counts, freq=None, ws=ws, ws_bytes=big):
        return handle.phm_kmer_count_spans(seq, off, n_rec, spans, n, k, flags, counts, freq, ws, ws_bytes, None)

    cases = [
        (dict(k=0), b"k must be 1..6"), (dict(k=7), b"k must be 1..6"),
        (dict(flags=lib.PHM_COUNT_NAIVE), b"flags"), (dict(flags=4), b"flags"),
        (dict(n_rec=-1), b"n_records"), (dict(n=-2), b"n_spans"),
        (dict(seq=None), b"null pointer"), (dict(off=None), b"null pointer"), (dict(spans=None), b"null pointer"),
        (dict(ws=None), b"null pointer"), (dict(counts=None), b"both outputs are null"),
        (dict(seq=ctypes.c_void_p((1 << 20) + 8)), b"16-byte aligned"),
        (dict(spans=ctypes.c_void_p((3 << 20) + 4)), b"misaligned"), (dict(freq=ctypes.c_void_p((7 << 20) + 2)), b"misaligned"),
        (dict(counts=ctypes.c_void_p((4 << 20) + 2)), b"misaligned"), (dict(off=ctypes.c_void_p((2 << 20) + 4)), b"misaligned"),
    ]
    for kw, msg in cases:
        assert call(**kw) == -1, kw
        assert msg in handle.phm_last_error(), (kw, handle.phm_last_error())
    # a workspace without one list item per span: the lower bound, checked before the device is touched
    need = handle.phm_kmer_count_spans_workspace_bytes(5, 0, 4, 0)
    assert call(ws_bytes=need - 256) == -3 and b"workspace too small" in handle.phm_last_error()
    assert call(ws_bytes=100) == -3
    assert call(n=0, seq=None, off=None, spans=None, counts=None, ws=None) == 0               # no span reads nothing


# ---------------------------------------------------------------------------------------------------------------------
# command line
# ---------------------------------------------------------------------------------------------------------------------
def test_cli_span_checks(lib, tmp_path):
    from phamers_b200 import phamer
    features = tmp_path / "only" / "contigs.csv"
    features.parent.mkdir()
    features.write_text("# K-mer count file\nc0,%s\n" % ",".join(["1"] * 256))
    bed = tmp_path / "a.bed"
    bed.write_text("c0\t0\t10\n")
    for argv in (["-features", str(features), "-spans", str(bed)], ["-in", str(features.parent), "-spans", str(bed)],
                 ["-fasta", "x.fasta", "-region_scores"], ["-features", str(features), "-region_scores"]):
        with pytest.raises(SystemExit) as exc:
            phamer.main(argv + ["-out", str(tmp_path / "out")])
        assert exc.value.code == 2, argv


def test_cli_span_files_and_unchanged_outputs(lib, monkeypatch, tmp_path):
    """-spans and -region_scores write their files; every file a run writes without them is byte for byte what it was."""
    from phamers_b200 import fileIO, phamer
    fasta = tmp_path / "x.fasta"
    fasta.write_text(">c0\nACGT\n>c1\nACGT\n")
    bed = tmp_path / "a.bed"
    bed.write_text("track x\nc1\t1\t3\tg1\nc0 0 2\n")

    def load_data(self, length_requirement=None):
        self.data_ids = np.array(["c0", "c1"])
        self.data_points = np.zeros((2, 256))

    def score_neighbors(self):
        self.neighbor_ids, self.neighbor_labels = np.array([["r1"], ["r2"]]), np.array([[1], [0]])
        self.neighbor_distances, self.nearest_clusters = np.array([[0.5], [0.25]]), np.array([[1, 2], [3, 4]])
        self.nearest_cluster_distances = np.array([[0.1, 0.2], [0.3, 0.4]])
        return np.array([0.5, -0.25])

    def score_windows(self, window, step=None):
        self.window_ids, self.window_records = np.array(["c0", "c0", "c1"]), np.array([0, 0, 1])
        self.window_spans = np.array([[0, window], [step, step + window], [0, 3]])
        self.window_scores = np.array([0.5, -0.25, 1.25])
        return self.window_scores

    def fill(self, scores):
        n = len(self.span_ids)
        self.span_scores = np.asarray(scores, dtype=np.float64)
        self.span_neighbor_ids, self.span_neighbor_labels = np.full((n, 1), "r9"), np.ones((n, 1), dtype=np.int64)
        self.span_neighbor_distances, self.span_nearest_clusters = np.full((n, 1), 0.75), np.zeros((n, 2), dtype=np.int64)
        self.span_nearest_cluster_distances = np.full((n, 2), 0.5)
        return self.span_scores

    def score_spans(self, ids, spans, names=None, lines=None):
        assert lines == ["%s line %d" % (bed, n) for n in (2, 3)]
        self.span_ids, self.span_spans, self.span_names = np.asarray(ids), np.asarray(spans), np.asarray(names)
        return fill(self, [0.125, -1.0])

    def score_regions(self):
        assert self.region_records.tolist() == [0, 1]
        self.span_ids, self.span_spans = self.region_ids, self.region_spans
        self.span_names = np.full((len(self.span_ids),), ".")
        return fill(self, np.arange(len(self.span_ids)) * 0.5)

    monkeypatch.setattr(phamer.phamer_scorer, "load_reference_data", lambda self, p=None, n=None: None)
    monkeypatch.setattr(phamer.phamer_scorer, "load_data", load_data)
    monkeypatch.setattr(phamer.phamer_scorer, "score_neighbors", score_neighbors)
    monkeypatch.setattr(phamer.phamer_scorer, "score_windows", score_windows)
    monkeypatch.setattr(phamer.phamer_scorer, "score_spans", score_spans)
    monkeypatch.setattr(phamer.phamer_scorer, "score_regions", score_regions)
    out = tmp_path / "out"                                               # the output directory is part of the headers
    base = ["-fasta", str(fasta), "-l", "0", "-out", str(out), "-neighbors", "-window", "100", "-step", "40"]
    phamer.main(base)
    names = ("phamer_scores.csv", "phamer_neighbors.csv", "phamer_windows.csv", "phamer_regions.csv")
    before = {n: open(out / n, "rb").read() for n in names}
    assert not (out / "phamer_spans.csv").exists() and not (out / "phamer_region_scores.csv").exists()
    phamer.main(base + ["-spans", str(bed), "-region_scores"])
    for n in names:
        assert open(out / n, "rb").read() == before[n], n
    s = fileIO.read_phamer_spans(str(out / "phamer_spans.csv"))
    assert s[0].tolist() == ["c1", "c0"] and s[1].tolist() == [[1, 3], [0, 2]] and s[2].tolist() == ["g1", "."]
    assert s[3].tolist() == [0.125, -1.0] and s[4].tolist() == [["r9"], ["r9"]]
    r = fileIO.read_phamer_regions(str(out / "phamer_regions.csv"))
    rs = fileIO.read_phamer_spans(str(out / "phamer_region_scores.csv"))
    assert np.array_equal(rs[0], r[0]) and np.array_equal(rs[1], r[1]) and rs[2].tolist() == ["."] * len(r[0])
    assert "span_file:\t" in open(out / "phamer_spans.csv").read()

"""CPU-only checks of sliding-window scoring: the window enumeration (closed form against the contract's loop), region finding on
hand-made scores, round trips of the window and region files, the argument errors of the window entry points (reported before a
device is touched), and the command line's checks and file plumbing."""
import ctypes
import math

import numpy as np
import pytest

import __graft_entry__ as entry


@pytest.fixture(scope="module")
def lib():
    entry.build()
    from phamers_b200 import _lib
    return _lib


# ---------------------------------------------------------------------------------------------------------------------
# the window contract
# ---------------------------------------------------------------------------------------------------------------------
def brute_windows(length, window, step):
    """The contract as stated: [j s, j s + w) while j s + w <= L, then one window aligned to the record end if the last ends before L."""
    if length <= window:
        return [(0, length)]
    out, j = [], 0
    while j * step + window <= length:
        out.append((j * step, j * step + window))
        j += 1
    if out[-1][1] < length:
        out.append((length - window, length))
    return out


def window_table(lengths, window, step):
    """Closed form used by the kernels: (window offsets int64[n + 1], spans int64[windows, 2] relative to the record)."""
    lengths = np.asarray(lengths, dtype=np.int64)
    counts = np.where(lengths <= window, 1, 2 + (lengths - window - 1) // step)
    wo = np.concatenate(([0], np.cumsum(counts))).astype(np.int64)
    spans = []
    for length, c in zip(lengths.tolist(), counts.tolist()):
        for j in range(c):
            a = 0 if length <= window else (j * step if j + 1 < c else length - window)
            spans.append((a, min(a + window, length) if length > window else length))
    return wo, np.array(spans, dtype=np.int64).reshape(-1, 2)


@pytest.mark.parametrize("window,step,k", [(10, 3, 4), (10, 10, 4), (10, 15, 4), (12, 4, 4), (3, 1, 4), (5000, 1000, 4), (7, 2, 6)])
def test_window_enumeration(window, step, k):
    lengths = {0, 1, k - 1, window - 1, window, window + 1, window + step - 1, window + step, window + step + 1}
    lengths |= {window + m * step for m in range(5)} | {window + m * step + r for m in range(3) for r in (1, step // 2)}
    lengths |= {2 * window + 1, 3 * window + step, 7 * step + 3}
    lengths = sorted(x for x in lengths if x >= 0)
    wo, spans = window_table(lengths, window, step)
    assert wo[0] == 0 and len(wo) == len(lengths) + 1
    for r, length in enumerate(lengths):
        want = brute_windows(length, window, step)
        got = [tuple(s) for s in spans[wo[r]:wo[r + 1]].tolist()]
        assert got == want, (length, window, step)
        if length > window:
            assert len(got) == 1 + math.ceil((length - window) / step)
            assert all(b - a == window for a, b in got)
            if step <= window:
                assert got[0][0] == 0 and got[-1][1] == length
                assert all(got[i + 1][0] <= got[i][1] for i in range(len(got) - 1))          # every base covered


# ---------------------------------------------------------------------------------------------------------------------
# regions
# ---------------------------------------------------------------------------------------------------------------------
def _regions(ids, records, spans, scores):
    from phamers_b200 import phamer
    sc = phamer.phamer_scorer()
    sc.window_ids, sc.window_records = np.asarray(ids), np.asarray(records)
    sc.window_spans, sc.window_scores = np.asarray(spans).reshape(-1, 2), np.asarray(scores, dtype=np.float64)
    sc.find_regions()
    return sc


def test_find_regions():
    nan = float("nan")
    # record 0: 6 windows with a NaN inside a positive run; record 1: one window; records 2 and 3 wholly positive and adjacent
    ids = ["a"] * 6 + ["b"] + ["c"] * 3 + ["d"] * 2
    records = [0] * 6 + [1] + [2] * 3 + [3] * 2
    spans = [(0, 10), (5, 15), (10, 20), (15, 25), (20, 30), (22, 32), (0, 7), (0, 10), (5, 15), (8, 18), (0, 10), (3, 13)]
    scores = [-0.5, 0.25, 1.5, nan, 0.0, 0.75, 0.5, 0.1, 0.2, 0.3, 1.0, 0.0]
    sc = _regions(ids, records, spans, scores)
    assert sc.region_ids.tolist() == ["a", "a", "b", "c", "d"]
    assert sc.region_spans.tolist() == [[5, 20], [20, 32], [0, 7], [0, 18], [0, 13]]
    assert sc.region_windows.tolist() == [2, 2, 1, 3, 2]
    assert np.allclose(sc.region_mean_scores, [0.875, 0.375, 0.5, 0.2, 0.5], rtol=0, atol=1e-15)
    assert sc.region_max_scores.tolist() == [1.5, 0.75, 0.5, 0.3, 1.0]
    # a single negative window, NaN only, nothing at all
    for s in ([-0.1], [nan], []):
        sc = _regions(["x"] * len(s), [0] * len(s), [(0, 5)] * len(s), s)
        assert len(sc.region_ids) == 0 and sc.region_spans.shape == (0, 2) and len(sc.region_mean_scores) == 0
    # one record wholly positive
    sc = _regions(["x"] * 4, [7] * 4, [(0, 4), (2, 6), (4, 8), (5, 9)], [0.5, 0.25, 0.125, 1.0])
    assert sc.region_spans.tolist() == [[0, 9]] and sc.region_windows.tolist() == [4] and sc.region_max_scores.tolist() == [1.0]
    # two records with the same id stay apart
    sc = _regions(["x", "x"], [0, 1], [(0, 5), (0, 5)], [0.5, 0.5])
    assert sc.region_windows.tolist() == [1, 1]


# ---------------------------------------------------------------------------------------------------------------------
# files
# ---------------------------------------------------------------------------------------------------------------------
def test_window_and_region_files_round_trip(tmp_path):
    from phamers_b200 import fileIO
    rng = np.random.default_rng(5)
    ids = np.array(["c%d" % i for i in rng.integers(0, 50, size=200)])
    spans = np.sort(rng.integers(0, 1 << 40, size=(200, 2)), axis=1)
    scores = rng.normal(size=200) * 10.0 ** rng.integers(-20, 3, size=200)
    scores[[3, 17]] = np.nan
    path = str(tmp_path / "w.csv")
    fileIO.save_phamer_windows(ids, spans, scores, path)
    r_ids, r_spans, r_scores = fileIO.read_phamer_windows(path)
    assert np.array_equal(r_ids, ids) and np.array_equal(r_spans, spans) and np.array_equal(r_scores, scores, equal_nan=True)
    text = open(path).read().splitlines()
    assert text[0] == "# PhaMers window file" and text[1] == "# id, start, end, score"
    windows = rng.integers(1, 100, size=200)
    mean, mx = rng.random(200), rng.random(200) * 1.7616
    path = str(tmp_path / "r.csv")
    fileIO.save_phamer_regions(ids, spans, windows, mean, mx, path)
    back = fileIO.read_phamer_regions(path)
    for a, b in zip(back, (ids, spans, windows, mean, mx)):
        assert np.array_equal(a, b)
    assert open(path).read().splitlines()[1] == "# id, start, end, windows, mean_score, max_score"
    fileIO.save_phamer_regions([], np.zeros((0, 2)), [], [], [], path)
    assert [len(a) for a in fileIO.read_phamer_regions(path)] == [0] * 5


# ---------------------------------------------------------------------------------------------------------------------
# argument errors of the entry points: reported through phm_last_error before any device is touched
# ---------------------------------------------------------------------------------------------------------------------
def test_window_symbols_load(lib):
    handle = lib.load()
    for name in ("phm_window_offsets", "phm_kmer_count_windows_workspace_bytes", "phm_kmer_count_windows"):
        assert getattr(handle, name).argtypes == lib.SIGNATURES[name][1]
    fixed = handle.phm_kmer_count_windows_workspace_bytes(0, 1, 4, 0)
    assert handle.phm_kmer_count_windows_workspace_bytes(1000, 5000, 4, 0) == fixed + 32000
    assert handle.phm_kmer_count_windows_workspace_bytes(1000, 300000, 4, 0) == fixed + 4 * 32000   # 300 000 bases: 4 tiles


def test_window_offsets_argument_errors(lib):
    handle = lib.load()
    off, wo = ctypes.c_void_p(256), ctypes.c_void_p(512)
    for w, s in ((0, 1), (1, 0), (-5, 3), (3, -1)):
        assert handle.phm_window_offsets(off, 4, w, s, wo, None) == -1
        assert b"window and step" in handle.phm_last_error()
    assert handle.phm_window_offsets(off, -1, 5, 5, wo, None) == -1 and b"n_records" in handle.phm_last_error()
    assert handle.phm_window_offsets(off, 4, 5, 5, None, None) == -1 and b"null pointer" in handle.phm_last_error()
    assert handle.phm_window_offsets(None, 4, 5, 5, wo, None) == -1 and b"null pointer" in handle.phm_last_error()
    assert handle.phm_window_offsets(ctypes.c_void_p(260), 4, 5, 5, wo, None) == -1 and b"aligned" in handle.phm_last_error()


def test_count_windows_argument_errors(lib):
    handle = lib.load()
    seq, off, wo, counts, ws = (ctypes.c_void_p(v) for v in (1 << 20, 2 << 20, 3 << 20, 4 << 20, 5 << 20))
    big = 1 << 30

    def call(seq=seq, off=off, n_rec=10, wo=wo, w=100, s=50, first=0, n=5, k=4, flags=0, counts=counts, freq=None, spans=None,
             ws=ws, ws_bytes=big):
        return handle.phm_kmer_count_windows(seq, off, n_rec, wo, w, s, first, n, k, flags, counts, freq, spans, ws, ws_bytes, None)

    cases = [
        (dict(k=0), b"k must be 1..6"), (dict(k=7), b"k must be 1..6"),
        (dict(w=0), b"window and step"), (dict(s=0), b"window and step"),
        (dict(flags=lib.PHM_COUNT_NAIVE), b"flags"), (dict(flags=4), b"flags"),
        (dict(n_rec=-1), b"n_records"), (dict(first=-1), b"first_window"), (dict(n=-2), b"n_windows"),
        (dict(n_rec=0), b"outside"),
        (dict(seq=None), b"null pointer"), (dict(off=None), b"null pointer"), (dict(wo=None), b"null pointer"),
        (dict(ws=None), b"null pointer"), (dict(counts=None), b"both outputs are null"),
        (dict(seq=ctypes.c_void_p((1 << 20) + 8)), b"16-byte aligned"),
        (dict(spans=ctypes.c_void_p((6 << 20) + 4)), b"misaligned"), (dict(freq=ctypes.c_void_p((7 << 20) + 2)), b"misaligned"),
        (dict(counts=ctypes.c_void_p((4 << 20) + 2)), b"misaligned"), (dict(wo=ctypes.c_void_p((3 << 20) + 4)), b"misaligned"),
    ]
    for kw, msg in cases:
        assert call(**kw) == -1, kw
        assert msg in handle.phm_last_error(), (kw, handle.phm_last_error())
    need = handle.phm_kmer_count_windows_workspace_bytes(5, 100, 4, 0)
    assert call(ws_bytes=need - 256) == -3 and b"workspace too small" in handle.phm_last_error()
    assert call(n=0, seq=None, off=None, wo=None, counts=None, ws=None) == 0                 # an empty slice reads nothing
    assert call(n_rec=0, n=0) == 0


# ---------------------------------------------------------------------------------------------------------------------
# command line
# ---------------------------------------------------------------------------------------------------------------------
def test_cli_window_checks(lib, tmp_path):
    from phamers_b200 import phamer
    features = tmp_path / "only" / "contigs.csv"
    features.parent.mkdir()
    features.write_text("# K-mer count file\nc0,%s\n" % ",".join(["1"] * 256))
    for argv in (["-features", str(features), "-window", "5000"], ["-in", str(features.parent), "-window", "5000"],
                 ["-fasta", "x.fasta", "-step", "10"], ["-fasta", "x.fasta", "-window", "0"],
                 ["-fasta", "x.fasta", "-window", "10", "-step", "0"]):
        with pytest.raises(SystemExit) as exc:
            phamer.main(argv + ["-out", str(tmp_path / "out")])
        assert exc.value.code == 2, argv


def test_cli_window_files_and_unchanged_score_file(lib, monkeypatch, tmp_path):
    """The window run writes both files; its score file is byte for byte that of the run without -window."""
    from phamers_b200 import fileIO, phamer
    fasta = tmp_path / "x.fasta"
    fasta.write_text(">c0\nACGT\n>c1\nACGT\n")

    def load_data(self, length_requirement=None):
        self.data_ids = np.array(["c0", "c1"])
        self.data_points = np.zeros((2, 256))

    def score_windows(self, window, step=None):
        self.window_ids = np.array(["c0", "c0", "c1"])
        self.window_records = np.array([0, 0, 1])
        self.window_spans = np.array([[0, window], [step, step + window], [0, 3]])
        self.window_scores = np.array([0.5, -0.25, 1.25])
        return self.window_scores

    monkeypatch.setattr(phamer.phamer_scorer, "load_reference_data", lambda self, p=None, n=None: None)
    monkeypatch.setattr(phamer.phamer_scorer, "load_data", load_data)
    monkeypatch.setattr(phamer.phamer_scorer, "score_points", lambda self: np.array([0.5, -0.25]))
    monkeypatch.setattr(phamer.phamer_scorer, "score_windows", score_windows)
    base = ["-fasta", str(fasta), "-l", "0", "-canonical"]
    out = tmp_path / "win"                                               # the output directory is part of the header
    phamer.main(base + ["-out", str(out)])
    plain = open(out / "phamer_scores.csv").read()
    assert not (out / "phamer_windows.csv").exists()
    phamer.main(base + ["-out", str(out), "-window", "100", "-step", "40"])
    assert open(out / "phamer_scores.csv").read() == plain
    ids, spans, scores = fileIO.read_phamer_windows(str(tmp_path / "win" / "phamer_windows.csv"))
    assert ids.tolist() == ["c0", "c0", "c1"] and spans.tolist() == [[0, 100], [40, 140], [0, 3]]
    r = fileIO.read_phamer_regions(str(tmp_path / "win" / "phamer_regions.csv"))
    assert r[0].tolist() == ["c0", "c1"] and r[1].tolist() == [[0, 100], [0, 3]] and r[2].tolist() == [1, 1]
    assert "window_length:\t100" in open(tmp_path / "win" / "phamer_windows.csv").read()

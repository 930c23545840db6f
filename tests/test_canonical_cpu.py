"""CPU-only checks of canonical (strand-independent) scoring: phm_canonical_fold reports argument errors through phm_last_error
before touching a device, the new symbols load, the command line checks the width of a features CSV, and the score file's header
is unchanged without -canonical."""
import argparse
import ctypes

import numpy as np
import pytest

import __graft_entry__ as entry


@pytest.fixture(scope="module")
def lib():
    entry.build()
    from phamers_b200 import _lib
    return _lib


def test_canonical_symbols_load(lib):
    handle = lib.load()
    assert "phm_canonical_fold" in lib.SIGNATURES
    assert handle.phm_canonical_fold.argtypes == lib.SIGNATURES["phm_canonical_fold"][1]
    assert [handle.phm_num_bins(4, lib.PHM_COUNT_CANONICAL), handle.phm_num_bins(4, 0)] == [136, 256]


def test_canonical_fold_argument_errors(lib):
    handle = lib.load()
    rows, out = ctypes.c_void_p(16), ctypes.c_void_p(16)
    for k in (0, 7):
        assert handle.phm_canonical_fold(rows, 4, k, out, None) == -1
        assert b"k must be 1..6" in handle.phm_last_error()
    assert handle.phm_canonical_fold(None, 4, 4, out, None) == -1 and b"null pointer" in handle.phm_last_error()
    assert handle.phm_canonical_fold(rows, 4, 4, None, None) == -1 and b"null pointer" in handle.phm_last_error()
    assert handle.phm_canonical_fold(rows, -1, 4, out, None) == -1 and b"n_rows" in handle.phm_last_error()
    assert handle.phm_canonical_fold(None, 0, 4, None, None) == 0          # nothing to fold: no pointer is read


def _write_features(path, width, n=3):
    with open(path, "w") as fh:
        fh.write("# K-mer count file\n")
        for i in range(n):
            fh.write("c%d,%s\n" % (i, ",".join(str((i + j) % 7) for j in range(width))))


def test_canonical_width_check(lib, tmp_path):
    from phamers_b200 import phamer
    scorer = phamer.phamer_scorer()
    scorer.canonical = True
    path = str(tmp_path / "features.csv")
    for width in (100, 255, 512):
        _write_features(path, width)
        scorer.features_file = path
        with pytest.raises(ValueError, match="canonical scoring at k = 4"):
            scorer.load_data(length_requirement=0)
    canon = np.arange(2 * 136).reshape(2, 136)
    assert scorer._features(canon) is canon                              # already canonical width: taken as it is
    scorer.canonical = False
    plain = np.ones((2, 100))
    assert scorer._features(plain) is plain                              # plain mode never looks at the width


def _score_file_header(monkeypatch, tmp_path, argv):
    from phamers_b200 import phamer

    def load_data(self, length_requirement=None):
        self.data_ids = np.array(["c0", "c1"])
        self.data_points = np.zeros((2, 256))
    monkeypatch.setattr(phamer.phamer_scorer, "load_reference_data", lambda self, p=None, n=None: None)
    monkeypatch.setattr(phamer.phamer_scorer, "load_data", load_data)
    monkeypatch.setattr(phamer.phamer_scorer, "score_points", lambda self: np.array([0.5, -0.25]))
    out = tmp_path / "out"
    scorer = phamer.main(argv + ["-out", str(out)])
    return open(out / "phamer_scores.csv").read(), scorer


def test_score_file_header_without_canonical(lib, monkeypatch, tmp_path):
    from phamers_b200 import fileIO
    text, scorer = _score_file_header(monkeypatch, tmp_path, ["-fasta", "x.fasta", "-l", "0"])
    assert scorer.canonical is False
    # the header of the parent version: every argument but write_neighbors, in the order they are declared
    want = argparse.Namespace(input_directory=None, fasta_file="x.fasta", features_file=None, data_directory=None,
                              positive_features=None, negative_features=None, output_directory=str(tmp_path / "out"),
                              kmer_length=4, length_requirement=0, equalize_reference=False, method="combo", do_tsne=False,
                              plot_tsne=False)
    assert "canonical" not in text
    fileIO.save_phamer_scores(np.array(["c0", "c1"]), np.array([0.5, -0.25]), str(tmp_path / "want.csv"), args=want)
    assert text == open(tmp_path / "want.csv").read()
    text, scorer = _score_file_header(monkeypatch, tmp_path, ["-fasta", "x.fasta", "-l", "0", "-canonical"])
    assert scorer.canonical is True and "canonical_kmers:\tTrue" in text

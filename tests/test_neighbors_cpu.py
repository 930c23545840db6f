"""CPU-only checks of the neighbour report: the neighbour file round-trips, and the new entry points report argument errors through
phm_last_error before touching a device."""
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


def test_neighbor_file_round_trip(tmp_path):
    from phamers_b200 import fileIO
    rng = np.random.default_rng(5)
    n, k = 7, 3
    ids = np.array(["contig_%d" % i for i in range(n)])
    refs = rng.choice(np.array(["NC_001416.1", "NZ_CP009072.1", "AB000001.2"]), size=(n, k))
    labels = rng.integers(0, 2, size=(n, k))
    dist = np.sort(rng.random((n, k)) * 0.1, axis=1)
    dist[0, 0] = 0.0
    dist[1] = np.nextafter(dist[1], 1.0)                     # last-bit values must survive the text form
    clusters = rng.integers(0, 86, size=(n, 2))
    cdist = rng.random((n, 2))
    refs[3], labels[3], dist[3], clusters[3], cdist[3] = "", -1, np.nan, -1, np.nan      # a contig with no countable k-mer
    args = argparse.Namespace(input_directory="sample", write_neighbors=True)
    path = str(tmp_path / "phamer_neighbors.csv")
    fileIO.save_phamer_neighbors(ids, refs, labels, dist, clusters, cdist, path, args=args)
    text = open(path).read()
    assert text.startswith("# PhaMers neighbour file\n# input_directory:\t'sample'\n")
    assert "# id, reference_1, class_1, distance_1, reference_2" in text
    assert "phage_cluster, phage_cluster_distance, bacteria_cluster, bacteria_cluster_distance\n" in text
    r_ids, r_refs, r_labels, r_dist, r_clusters, r_cdist = fileIO.read_phamer_neighbors(path)
    assert list(r_ids) == list(ids)
    assert np.array_equal(r_refs, refs) and np.array_equal(r_labels, labels) and np.array_equal(r_clusters, clusters)
    assert np.array_equal(r_dist, dist, equal_nan=True) and np.array_equal(r_cdist, cdist, equal_nan=True)
    row0 = [line for line in text.splitlines() if line.startswith("contig_0, ")][0].split(", ")
    assert row0[2] in ("phage", "bacteria") and len(row0) == 1 + 3 * k + 4


def _score_neighbors(handle, points, n_points, k, nb):
    return handle.phm_score_neighbors(points, n_points, 256, ctypes.c_void_p(16), 10, 5, None, 0, None, 0, k,
                                      None, None, None, ctypes.byref(nb), ctypes.c_void_p(16), 1 << 20, None)


def test_neighbor_entry_points_report_argument_errors(lib):
    handle = lib.load()
    nb = lib.Neighbors()
    for k in (0, 16, 11):                                    # 1..15 and at most n_refs (10)
        rc = _score_neighbors(handle, ctypes.c_void_p(16), 4, k, nb)
        assert rc == -1 and b"k_neighbors must be 1..15" in handle.phm_last_error()
    rc = _score_neighbors(handle, None, 4, 3, nb)
    assert rc == -1 and b"d_points is null" in handle.phm_last_error()
    rc = handle.phm_score_counts_neighbors(None, 4, 256, ctypes.c_void_p(16), 10, 5, None, 0, None, 0, 3,
                                           None, None, None, ctypes.byref(nb), ctypes.c_void_p(16), 1 << 20, None)
    assert rc == -1 and b"d_counts is null" in handle.phm_last_error()
    rc = handle.phm_score_counts_neighbors(ctypes.c_void_p(16), 4, 256, ctypes.c_void_p(16), 10, 5, None, 0, None, 0, 0,
                                           None, None, None, None, ctypes.c_void_p(16), 1 << 20, None)
    assert rc == -1 and b"k_neighbors must be 1..15" in handle.phm_last_error()
    assert _score_neighbors(handle, None, 0, 3, nb) == 0   # nothing to score: no pointer is read

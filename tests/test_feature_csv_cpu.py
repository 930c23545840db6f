"""The feature CSV calls without a device: argument errors and workspace sizes of phm_counts_csv_* / phm_feature_csv_*, which come
back before the device is touched, and save_counts / read_feature_file on a machine without CUDA, which take the host road and
write and read what they always did."""
import ctypes

import numpy as np
import pytest

import __graft_entry__ as entry
from phamers_b200 import fileIO

PHM_E_ARG, PHM_E_WORKSPACE = -1, -3
FAKE = ctypes.c_void_p(1 << 20)            # a 16-byte aligned address that the calls must not dereference on these paths


@pytest.fixture(scope="module")
def lib():
    entry.build()
    from phamers_b200 import _lib
    return _lib.load()


def test_workspace_sizes(lib):
    for fn, unit in ((lib.phm_counts_csv_workspace_bytes, 256), (lib.phm_feature_csv_workspace_bytes, 4096)):
        sizes = [fn(n) for n in (0, 1, unit, unit + 1, 1000 * unit)]
        assert sizes == sorted(sizes) and all(s % 256 == 0 and s >= 256 for s in sizes)
        assert fn(1000 * unit) >= 1000 * 8                        # one int64 per tile at least
        assert fn(-5) == fn(0)


def test_format_argument_errors(lib):
    ws = lib.phm_counts_csv_workspace_bytes(10)
    layout = lib.phm_counts_csv_layout
    assert layout(FAKE, -1, 4, FAKE, 0, FAKE, FAKE, ws, None) == PHM_E_ARG
    assert layout(FAKE, 10, -4, FAKE, 0, FAKE, FAKE, ws, None) == PHM_E_ARG
    assert layout(FAKE, 10, 4, FAKE, -1, FAKE, FAKE, ws, None) == PHM_E_ARG
    assert layout(None, 10, 4, FAKE, 0, FAKE, FAKE, ws, None) == PHM_E_ARG
    assert layout(FAKE, 10, 4, None, 0, FAKE, FAKE, ws, None) == PHM_E_ARG
    assert layout(FAKE, 10, 4, FAKE, 0, None, FAKE, ws, None) == PHM_E_ARG
    assert layout(FAKE, 10, 4, FAKE, 0, FAKE, None, ws, None) == PHM_E_ARG
    assert layout(FAKE, 10, 4, FAKE, 0, FAKE, FAKE, ws - 1, None) == PHM_E_WORKSPACE
    assert b"workspace too small" in lib.phm_last_error()
    fmt = lib.phm_counts_csv_format
    assert fmt(FAKE, 10, 4, FAKE, FAKE, 5, FAKE, ctypes.c_void_p((1 << 20) + 8), 100, None) == PHM_E_ARG      # misaligned text
    assert b"16-byte aligned" in lib.phm_last_error()
    assert fmt(FAKE, 10, 4, None, FAKE, 5, FAKE, FAKE, 100, None) == PHM_E_ARG
    assert fmt(FAKE, 10, 4, FAKE, FAKE, 5, FAKE, None, 100, None) == PHM_E_ARG
    assert fmt(FAKE, 10, 4, FAKE, FAKE, 5, FAKE, FAKE, -1, None) == PHM_E_ARG
    assert fmt(FAKE, 10, 4, FAKE, None, 5, FAKE, FAKE, 100, None) == PHM_E_ARG


def test_parse_argument_errors(lib):
    ws = lib.phm_feature_csv_workspace_bytes(1000)
    index, parse = lib.phm_feature_csv_index, lib.phm_feature_csv_parse
    assert index(FAKE, -1, FAKE, FAKE, ws, None) == PHM_E_ARG
    assert index(FAKE, 1 << 40, FAKE, FAKE, 1 << 40, None) == PHM_E_ARG
    assert index(None, 1000, FAKE, FAKE, ws, None) == PHM_E_ARG
    assert index(FAKE, 1000, None, FAKE, ws, None) == PHM_E_ARG
    assert index(FAKE, 1000, FAKE, None, ws, None) == PHM_E_ARG
    assert index(ctypes.c_void_p((1 << 20) + 4), 1000, FAKE, FAKE, ws, None) == PHM_E_ARG
    assert index(FAKE, 1000, FAKE, FAKE, ws - 1, None) == PHM_E_WORKSPACE
    assert parse(FAKE, 1000, FAKE, FAKE, -1, 3, FAKE, ws, None) == PHM_E_ARG
    assert parse(FAKE, 1000, FAKE, FAKE, 5, -3, FAKE, ws, None) == PHM_E_ARG
    assert parse(FAKE, 1000, None, FAKE, 5, 3, FAKE, ws, None) == PHM_E_ARG
    assert parse(FAKE, 1000, FAKE, None, 5, 3, FAKE, ws, None) == PHM_E_ARG
    assert parse(FAKE, 1000, FAKE, FAKE, 5, 3, None, ws, None) == PHM_E_ARG
    assert parse(FAKE, 1000, FAKE, FAKE, 5, 3, FAKE, ws - 1, None) == PHM_E_WORKSPACE


@pytest.fixture
def no_device(monkeypatch):
    import torch
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)


def test_host_road_without_a_device(tmp_path, no_device):
    """The same text as the reference writes, read back into the same arrays, with no device anywhere."""
    path = str(tmp_path / "f.csv")
    counts = np.array([[0, -1, 12], [2 ** 63 - 1, -2 ** 63, 7]])
    fileIO.save_counts(counts, ["a b", "x,y"], path)
    assert open(path, "rb").read() == (b"# K-mer count file\na b,0,-1,12\nx,y,9223372036854775807,-9223372036854775808,7\n")
    fileIO.save_counts(np.arange(3), ["solo", "ignored"], path, header="h1\nh2")
    assert open(path, "rb").read() == b"# h1\n# h2\nsolo,0,1,2\n"
    open(path, "w").write("# c\n a , 1,+2 ,003 # tail\n\nb,4,-5,6\n")
    ids, rows = fileIO.read_feature_file(path)
    want_ids, want_rows = fileIO._read_feature_file_host(path)
    assert ids.tolist() == want_ids.tolist() == ["a ", "b"]
    assert rows.dtype == np.int64 and np.array_equal(rows, want_rows) and rows.tolist() == [[1, 2, 3], [4, -5, 6]]
    assert np.array_equal(fileIO.read_feature_file(path, id="b"), [[4, -5, 6]])
    open(path, "w").write("a,1\nb,1,2\n")
    with pytest.raises(ValueError):
        fileIO.read_feature_file(path)

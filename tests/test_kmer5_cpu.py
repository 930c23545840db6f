"""CPU-only checks of the 5-mer widths on the scoring boundary: argument errors name the widths the tensor-core road takes (256, 136,
512, 1024) and are reported before any device is touched, the workspace grows with the operand width, and ContigScorer refuses
reference rows of the wrong width for k = 5."""
import ctypes

import pytest

import __graft_entry__ as entry

FAKE = ctypes.c_void_p(1 << 20)          # never dereferenced: every call below fails its argument checks first


@pytest.fixture(scope="module")
def lib():
    entry.build()
    from phamers_b200 import _lib
    return _lib


def _score(handle, entry_name, dim, ws_bytes):
    fn = getattr(handle, entry_name)
    return fn(FAKE, 10, dim, FAKE, 8, 4, FAKE, 2, FAKE, 2, 3, FAKE, FAKE, FAKE, FAKE, ws_bytes, None)


def test_unsupported_widths_name_the_supported_set(lib):
    handle = lib.load()
    for dim in (64, 300, 2080, 4096):
        ws = handle.phm_score_workspace_bytes(10, 8, 2, 2, dim)
        rc = _score(handle, "phm_score_counts", dim, ws)
        assert rc != 0
        msg = handle.phm_last_error()
        assert b"256, 136, 512 or 1024" in msg, (dim, msg)
        try:
            lib.set_option("score_path", 2)
            rc = _score(handle, "phm_score", dim, ws)
            assert rc != 0 and b"256, 136, 512 or 1024" in handle.phm_last_error(), dim
        finally:
            lib.set_option("score_path", 0)


def test_workspace_follows_the_operand_width(lib):
    handle = lib.load()
    n, r = 100000, 4000
    at = {dim: handle.phm_score_workspace_bytes(n, r, 86, 86, dim) for dim in (136, 256, 512, 1024)}
    assert at[136] == at[256]                                           # canonical 4-mers use 256-wide operands
    # FP16 query operands of 2 (resp. 1) KB per row instead of 512 bytes, and the reference operands with them
    assert at[512] - at[256] >= n * 512 and at[1024] - at[512] >= n * 1024
    exact = (n + r + 86 + 86 + 8) * 8
    assert handle.phm_score_workspace_bytes(n, r, 86, 86, 64) == exact


def test_contig_scorer_checks_the_reference_width(lib, monkeypatch):
    import numpy as np
    from phamers_b200 import _lib, pipeline
    monkeypatch.setattr(_lib, "require_cuda", lambda: _lib.load())
    with pytest.raises(ValueError, match="k = 5 needs 1024"):
        pipeline.ContigScorer(np.ones((4, 256)) / 256, np.ones((4, 256)) / 256, kmer_length=5, centroids=(np.ones((1, 256)), np.ones((1, 256))))
    with pytest.raises(ValueError, match="k = 5 canonical needs 512"):
        pipeline.ContigScorer(np.ones((4, 1024)) / 1024, np.ones((4, 1024)) / 1024, kmer_length=5, canonical=True,
                              centroids=(np.ones((1, 1024)), np.ones((1, 1024))))

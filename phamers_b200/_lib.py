"""ctypes binding of libphamers_b200.so (the C-ABI of include/phamers_b200.h).  No fallbacks: a missing library or
device is an error."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# PHAMERS_B200_LIB: another build of the same library (tuning experiments only; it must export the same C-ABI)
_PATH = os.environ.get("PHAMERS_B200_LIB") or os.path.join(_HERE, "lib", "libphamers_b200.so")
_lib = None

PHM_COUNT_CANONICAL = 1
PHM_COUNT_NAIVE = 2

c_void_p, c_int, c_int64, c_uint32, c_uint64, c_size_t = (ctypes.c_void_p, ctypes.c_int, ctypes.c_int64,
                                                           ctypes.c_uint32, ctypes.c_uint64, ctypes.c_size_t)

# every symbol include/phamers_b200.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "phm_version": (c_int, []),
    "phm_last_error": (ctypes.c_char_p, []),
    "phm_device_caps": (c_int, [c_void_p]),
    "phm_set_option": (c_int, [ctypes.c_char_p, c_int64]),
    "phm_num_bins": (c_int64, [c_int, c_uint32]),
    "phm_pack_fasta": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "phm_kmer_count_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int, c_uint32]),
    "phm_kmer_count": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_uint32, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "phm_window_offsets": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p]),
    "phm_kmer_count_windows_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int, c_uint32]),
    "phm_kmer_count_windows": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64, c_int64, c_int, c_uint32,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "phm_kmer_count_spans_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int, c_uint32]),
    "phm_kmer_count_spans": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_int, c_uint32, c_void_p, c_void_p, c_void_p,
                                     c_size_t, c_void_p]),
    "phm_kmer_count_packed": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_uint32, c_void_p, c_void_p,
                                      c_void_p, c_size_t, c_void_p]),
    "phm_canonical_fold": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "phm_normalize_counts": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "phm_normalize_rows": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "phm_distances": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "phm_kernel_launches": (c_uint64, []),
    "phm_score_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int64, c_int]),
    "phm_score": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_int64,
                          c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "phm_score_counts": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_int64,
                                 c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "phm_score_neighbors": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_int64,
                                    c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "phm_score_counts_neighbors": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p,
                                           c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "phm_count_score_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int64, c_int64]),
    "phm_count_score": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_int64,
                                c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "phm_score_stats": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "phm_kmeans_workspace_bytes": (c_size_t, [c_int64, c_int, c_int]),
    "phm_kmeans_lloyd": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int, c_int, ctypes.c_double, c_void_p, c_void_p, c_void_p, c_size_t,
                                 c_void_p]),
    "phm_fasta_workspace_bytes": (c_size_t, [c_int64]),
    "phm_fasta_index": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_size_t, c_void_p]),
    "phm_fasta_extract": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_size_t, c_void_p]),
    "phm_inflate_workspace_bytes": (c_size_t, [c_int64]),
    "phm_inflate": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_size_t, c_void_p]),
    "phm_gunzip_index_workspace_bytes": (c_size_t, [c_int64]),
    "phm_gunzip_index": (c_int, [c_void_p, c_int64, c_uint32, c_void_p, c_void_p, c_size_t, c_void_p]),
    "phm_gunzip_extract_workspace_bytes": (c_size_t, [c_int64]),
    "phm_gunzip_extract": (c_int, [c_void_p, c_int64, c_uint32, c_void_p, c_size_t, c_void_p, c_int64, c_void_p, c_size_t, c_void_p]),
    "phm_counts_csv_workspace_bytes": (c_size_t, [c_int64]),
    "phm_counts_csv_layout": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_size_t, c_void_p]),
    "phm_counts_csv_format": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p]),
    "phm_feature_csv_workspace_bytes": (c_size_t, [c_int64]),
    "phm_feature_csv_index": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_size_t, c_void_p]),
    "phm_feature_csv_parse": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_size_t, c_void_p]),
    "phm_last_kernel_ms": (c_int, [ctypes.c_char_p, c_void_p]),
    "phm_synth_lengths": (c_int, [c_uint64, c_int64, c_int64, c_void_p, c_void_p]),
    "phm_synth_bases": (c_int, [c_uint64, c_int64, c_int64, c_void_p, c_void_p, c_void_p]),
}


class PhamersLibraryError(RuntimeError):
    pass


class PhamersDataError(PhamersLibraryError):
    """PHM_E_DATA: the input data is corrupt (phm_inflate: a member failed to decode; phm_gunzip_index / phm_gunzip_extract: the
    stream does not decode, or its CRC32, ISIZE or end differ from the trailer's)."""


PHM_E_DATA = -5


class Neighbors(ctypes.Structure):
    """phm_neighbors: device pointers of the neighbour report (NULL = not wanted)."""
    _fields_ = [("d_ref_index", c_void_p), ("d_ref_distance", c_void_p), ("d_centroid_index", c_void_p),
                ("d_centroid_distance", c_void_p)]


class Caps(ctypes.Structure):
    _fields_ = [("device", ctypes.c_int32), ("sm_major", ctypes.c_int32), ("sm_minor", ctypes.c_int32),
                ("sm_count", ctypes.c_int32), ("max_smem_optin", ctypes.c_int32), ("hbm_bytes", ctypes.c_int64)]


def path():
    return _PATH


def load():
    """dlopen the library and bind every declared symbol (no GPU needed for this)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_PATH):
        raise PhamersLibraryError(
            "%s is missing: run `python __graft_entry__.py` (nvcc, sm_100a) first; there is no CPU fallback" % _PATH)
    import torch  # noqa: F401  (brings the CUDA runtime shared object into the process; the library links against it)
    lib = ctypes.CDLL(_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as exc:
            raise PhamersLibraryError("%s does not export %s" % (_PATH, name)) from exc
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().phm_last_error()
        raise (PhamersDataError if rc == PHM_E_DATA else PhamersLibraryError)("libphamers_b200 error %d: %s" % (rc, msg.decode("utf-8", "replace") if msg else ""))


def require_cuda():
    """Loads the library and makes sure a CUDA device is usable; raises otherwise."""
    import torch
    lib = load()
    if not torch.cuda.is_available():
        raise PhamersLibraryError("phamers_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return lib


def device_caps():
    lib = require_cuda()
    caps = Caps()
    check(lib.phm_device_caps(ctypes.byref(caps)))
    return caps


def set_option(name, value):
    check(load().phm_set_option(name.encode(), int(value)))


def stream_ptr():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)

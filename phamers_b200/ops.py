"""
Tensor-native host layer over the C-ABI: device tensors in, device tensors out, everything on the current CUDA
stream.  PyTorch is used for device memory and streams only; all arithmetic happens inside libphamers_b200.so.
The drop-in modules (kmer.py, phamer.py) convert to the reference's NumPy dtypes on top of these.
"""
import ctypes

import torch

from . import _lib
from ._lib import check, ptr, stream_ptr

_workspaces = {}
_last_score_ws = [None]      # the workspace the last scoring call used (score_stats reads its header)


def kernel_launches():
    """Kernels libphamers_b200.so has launched in this process (counted inside the library, one per <<< >>>)."""
    return int(_lib.load().phm_kernel_launches())


def _workspace(kind, nbytes):
    """Scratch memory of one call.  A workspace holds live kernel state (work counters, candidate lists), so it is private to
    (kind, device, STREAM): calls in flight on different streams never share one."""
    key = (kind, torch.cuda.current_device(), torch.cuda.current_stream().cuda_stream)
    buf = _workspaces.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 1 << 16), dtype=torch.uint8, device="cuda")
        _workspaces[key] = buf
    return buf


def _check(t, name, dtype, width=None):
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == dtype):
        raise TypeError("%s must be a CUDA %s tensor" % (name, dtype))
    if width is not None and (t.dim() != 2 or t.shape[1] != width):
        raise ValueError("%s must be [rows, %d]" % (name, width))
    return t.contiguous()


def _as_u8_cuda(seq):
    """The kernels read the sequence with 128-bit loads: 16-byte aligned start, storage readable up to the next multiple of 16."""
    if not (isinstance(seq, torch.Tensor) and seq.is_cuda and seq.dtype == torch.uint8 and seq.is_contiguous()):
        raise TypeError("sequence buffer must be a contiguous CUDA uint8 tensor")
    if seq.data_ptr() % 16:
        raise ValueError("sequence buffer must be 16-byte aligned")
    readable = seq.untyped_storage().nbytes() - seq.storage_offset()
    if readable < (seq.numel() + 15) // 16 * 16:
        raise ValueError("sequence storage must be readable up to the next multiple of 16 bytes (allocate %d more bytes)"
                         % ((seq.numel() + 15) // 16 * 16 - readable))
    return seq


def _result(given, shape, dtype):
    if given is None:
        return torch.empty(shape, dtype=dtype, device="cuda")
    if not (given.is_cuda and given.dtype == dtype and tuple(given.shape) == tuple(shape) and given.is_contiguous()):
        raise TypeError("preallocated result must be a contiguous CUDA %s tensor of shape %s" % (dtype, tuple(shape)))
    return given


def num_bins(k, canonical=False):
    n = _lib.load().phm_num_bins(int(k), _lib.PHM_COUNT_CANONICAL if canonical else 0)
    if n < 0:
        raise ValueError("k must be 1..6")
    return int(n)


def count_cuda(seq, offsets, k, canonical=False, counts=True, freq=False, naive=False, out_counts=None, out_freq=None):
    """K2+K3.  seq: uint8[total bases] (contigs end to end), offsets: int64[n+1].  Returns (counts int32[n, bins] or
    None, freq float64[n, bins] or None).  Counts are exact unsigned 32-bit values (< 2^31 for any contig this
    library accepts), stored in an int32 tensor because torch has no first-class uint32.  out_counts / out_freq: optional
    preallocated result tensors (int32 / float64 [n, bins]) for callers that score batch after batch."""
    lib = _lib.require_cuda()
    seq = _as_u8_cuda(seq)
    if not (offsets.is_cuda and offsets.dtype == torch.int64 and offsets.is_contiguous()):
        raise TypeError("offsets must be a contiguous CUDA int64 tensor")
    n = offsets.numel() - 1
    flags = (_lib.PHM_COUNT_CANONICAL if canonical else 0) | (_lib.PHM_COUNT_NAIVE if naive else 0)
    bins = num_bins(k, canonical)
    out_counts = _result(out_counts, (n, bins), torch.int32) if (counts or naive) else None
    out_freq = _result(out_freq, (n, bins), torch.float64) if freq else None
    ws_bytes = lib.phm_kmer_count_workspace_bytes(n, seq.numel(), int(k), flags)
    ws = _workspace("count", ws_bytes)
    check(lib.phm_kmer_count(ptr(seq), ptr(offsets), n, int(k), flags, ptr(out_counts), ptr(out_freq),
                             ptr(ws), ws.numel(), stream_ptr()))
    return (out_counts if counts else None), out_freq


def _offsets_cuda(offsets):
    if not (isinstance(offsets, torch.Tensor) and offsets.is_cuda and offsets.dtype == torch.int64 and offsets.is_contiguous()):
        raise TypeError("offsets must be a contiguous CUDA int64 tensor")
    return offsets


def window_offsets_cuda(offsets, window, step):
    """phm_window_offsets: int64[n+1] record offsets -> int64[n+1] window offsets (entry 0 = 0; record r owns windows
    [wo[r], wo[r+1])).  A record of length L has one window when L <= window, else 1 + ceil((L - window) / step)."""
    lib = _lib.require_cuda()
    offsets = _offsets_cuda(offsets)
    n = offsets.numel() - 1
    wo = torch.empty((n + 1,), dtype=torch.int64, device="cuda")
    check(lib.phm_window_offsets(ptr(offsets), n, int(window), int(step), ptr(wo), stream_ptr()))
    return wo


def count_windows_cuda(seq, offsets, window_offsets, window, step, k, first=0, n=None, canonical=False, counts=True, freq=False,
                       spans=False, out_counts=None):
    """phm_kmer_count_windows: k-mer counts of the windows [first, first + n) (n = None: to the last window; reading that number
    synchronises) into rows 0 .. n - 1.  Returns (counts int32[n, bins] or None, freq float64[n, bins] or None, spans int64[n, 2]
    (start, end relative to the record) or None).  The call reads the total number of windows from the device once, to check the
    slice."""
    lib = _lib.require_cuda()
    seq = _as_u8_cuda(seq)
    offsets, window_offsets = _offsets_cuda(offsets), _offsets_cuda(window_offsets)
    n_records = offsets.numel() - 1
    if window_offsets.numel() != n_records + 1:
        raise ValueError("window_offsets must have one entry more than there are records")
    if n is None:
        n = int(window_offsets[-1].item()) - int(first)
    if int(first) < 0 or n < 0:
        raise ValueError("the slice [%d, %d + %d) is not a range of windows" % (int(first), int(first), n))
    flags = _lib.PHM_COUNT_CANONICAL if canonical else 0
    bins = num_bins(k, canonical)
    out_counts = _result(out_counts, (n, bins), torch.int32) if counts else None
    out_freq = torch.empty((n, bins), dtype=torch.float64, device="cuda") if freq else None
    out_spans = torch.empty((n, 2), dtype=torch.int64, device="cuda") if spans else None
    ws = _workspace("count", lib.phm_kmer_count_windows_workspace_bytes(n, int(window), int(k), flags))
    check(lib.phm_kmer_count_windows(ptr(seq), ptr(offsets), n_records, ptr(window_offsets), int(window), int(step), int(first), int(n),
                                     int(k), flags, ptr(out_counts), ptr(out_freq), ptr(out_spans), ptr(ws), ws.numel(), stream_ptr()))
    return out_counts, out_freq, out_spans


def count_spans_cuda(seq, offsets, spans, k, canonical=False, counts=True, freq=False, out_counts=None):
    """phm_kmer_count_spans: k-mer counts of arbitrary spans of the records.  spans: int64 CUDA tensor [n, 3] of (record, start, end),
    0-based half-open in the record, in any order.  Row i holds span i: the counts of count_cuda on those bases as a record of their
    own (a span without a countable k-mer has a NaN feature row).  Returns (counts int32[n, bins] or None, freq float64[n, bins] or
    None).  The call validates the spans on the device and synchronises once; an invalid span raises PhamersLibraryError naming
    the lowest such index."""
    lib = _lib.require_cuda()
    seq = _as_u8_cuda(seq)
    offsets = _offsets_cuda(offsets)
    if not (isinstance(spans, torch.Tensor) and spans.is_cuda and spans.dtype == torch.int64 and spans.dim() == 2
            and spans.shape[1] == 3):
        raise TypeError("spans must be a CUDA int64 tensor [n, 3] of (record, start, end)")
    spans = spans.contiguous()
    n = spans.shape[0]
    flags = _lib.PHM_COUNT_CANONICAL if canonical else 0
    bins = num_bins(k, canonical)
    out_counts = _result(out_counts, (n, bins), torch.int32) if counts else None
    out_freq = torch.empty((n, bins), dtype=torch.float64, device="cuda") if freq else None
    # the summed span length bounds the tiles of the list; an invalid span may make it meaningless, and the device check reports it
    span_bases = int((spans[:, 2] - spans[:, 1]).clamp(min=0).sum().item()) if n else 0
    ws = _workspace("count", lib.phm_kmer_count_spans_workspace_bytes(n, span_bases, int(k), flags))
    check(lib.phm_kmer_count_spans(ptr(seq), ptr(offsets), offsets.numel() - 1, ptr(spans), n, int(k), flags, ptr(out_counts),
                                   ptr(out_freq), ptr(ws), ws.numel(), stream_ptr()))
    return out_counts, out_freq


def pack_cuda(seq):
    """K1.  uint8[n] ASCII -> (codes int32[ceil(n/16)], valid int32[ceil(n/32)])."""
    lib = _lib.require_cuda()
    seq = _as_u8_cuda(seq)
    n = seq.numel()
    codes = torch.empty(((n + 15) // 16,), dtype=torch.int32, device="cuda")
    valid = torch.empty(((n + 31) // 32,), dtype=torch.int32, device="cuda")
    check(lib.phm_pack_fasta(ptr(seq), n, ptr(codes), ptr(valid), stream_ptr()))
    return codes, valid


def count_packed_cuda(codes, valid, offsets, k, canonical=False, counts=True, freq=False):
    lib = _lib.require_cuda()
    n = offsets.numel() - 1
    flags = _lib.PHM_COUNT_CANONICAL if canonical else 0
    bins = num_bins(k, canonical)
    out_counts = torch.empty((n, bins), dtype=torch.int32, device="cuda") if counts else None
    out_freq = torch.empty((n, bins), dtype=torch.float64, device="cuda") if freq else None
    ws = _workspace("count", lib.phm_kmer_count_workspace_bytes(n, 0, int(k), flags))
    check(lib.phm_kmer_count_packed(ptr(codes), ptr(valid), ptr(offsets), n, int(k), flags, ptr(out_counts),
                                    ptr(out_freq), ptr(ws), ws.numel(), stream_ptr()))
    return out_counts, out_freq


def canonical_fold_cuda(rows, k):
    """Canonical fold of rows that already exist (phm_canonical_fold): float64[n, 4^k] -> float64[n, num_bins(k, canonical=True)], the
    bins and order of count_cuda(..., canonical=True).  Integer-valued rows below 2^53 fold exactly."""
    lib = _lib.require_cuda()
    rows = _check(rows, "rows", torch.float64, 4 ** int(k) if 1 <= int(k) <= 6 else None)
    out = torch.empty((rows.shape[0], num_bins(k, canonical=True)), dtype=torch.float64, device="cuda")
    check(lib.phm_canonical_fold(ptr(rows), rows.shape[0], int(k), ptr(out), stream_ptr()))
    return out


def normalize_cuda(counts):
    """kmer.normalize_counts on the device: int32/uint32[n, bins] -> float64[n, bins]."""
    lib = _lib.require_cuda()
    if counts.dtype != torch.int32 or not counts.is_cuda:
        raise TypeError("counts must be a CUDA int32 tensor")
    counts = counts.contiguous()
    two_d = counts.reshape(-1, counts.shape[-1])
    out = torch.empty(two_d.shape, dtype=torch.float64, device="cuda")
    check(lib.phm_normalize_counts(ptr(two_d), two_d.shape[0], two_d.shape[1], ptr(out), stream_ptr()))
    return out.reshape(counts.shape)


def normalize_rows_cuda(rows):
    """kmer.normalize_counts for rows that are not exact 32-bit counts: float64[n, bins] (or [bins]) -> row / row sum."""
    lib = _lib.require_cuda()
    rows = _check(rows, "rows", torch.float64)
    two_d = rows.reshape(-1, rows.shape[-1])
    out = torch.empty_like(two_d)
    check(lib.phm_normalize_rows(ptr(two_d), two_d.shape[0], two_d.shape[1], ptr(out), stream_ptr()))
    return out.reshape(rows.shape)


def distances_cuda(point, rows):
    """learning.distances: float64 Euclidean distance of point[dim] to every row of rows[n, dim]."""
    lib = _lib.require_cuda()
    point, rows = _check(point, "point", torch.float64), _check(rows, "rows", torch.float64)
    if rows.dim() != 2 or point.numel() != rows.shape[1]:
        raise ValueError("point must have as many elements as rows has columns")
    out = torch.empty((rows.shape[0],), dtype=torch.float64, device="cuda")
    check(lib.phm_distances(ptr(point), ptr(rows), rows.shape[0], rows.shape[1], ptr(out), stream_ptr()))
    return out


def score_cuda(points, refs, n_positive, cent_pos, cent_neg, k_neighbors=3, out=None):
    """K4+K5.  float64 CUDA tensors: points[n, d], refs[R, d] (positives first), centroids[C, d].
    `points` may also be the int32 count matrix of count_cuda: the features (count / row total) are then formed on the fly
    inside the kernels and never materialised (tensor-core shapes only).
    Returns (knn, kmeans, combo) float64[n]; out = optional preallocated (knn, kmeans, combo)."""
    lib = _lib.require_cuda()
    points, refs, cent_pos, cent_neg = _score_inputs(points, refs, cent_pos, cent_neg)
    n, dim = points.shape
    knn, kmeans, combo = (_result(t, (n,), torch.float64) for t in (out if out is not None else (None, None, None)))
    ws = _score_workspace(lib, points, refs, cent_pos, cent_neg)
    entry = lib.phm_score_counts if points.dtype == torch.int32 else lib.phm_score
    check(entry(ptr(points), n, dim, ptr(refs), refs.shape[0], int(n_positive),
                ptr(cent_pos), cent_pos.shape[0], ptr(cent_neg), cent_neg.shape[0], int(k_neighbors),
                ptr(knn), ptr(kmeans), ptr(combo), ptr(ws), ws.numel(), stream_ptr()))
    return knn, kmeans, combo


def _score_inputs(points, refs, cent_pos, cent_neg):
    from_counts = points.dtype == torch.int32
    tensors = [points, refs, cent_pos, cent_neg]
    for t in tensors[1:] if from_counts else tensors:
        if not (t.is_cuda and t.dtype == torch.float64):
            raise TypeError("score_cuda takes CUDA float64 tensors (queries may be int32 counts)")
    if not points.is_cuda:
        raise TypeError("score_cuda takes CUDA tensors")
    points, refs, cent_pos, cent_neg = (t.contiguous() for t in tensors)
    dim = points.shape[1]
    if refs.shape[1] != dim or (cent_pos.numel() and cent_pos.shape[1] != dim) or (cent_neg.numel() and cent_neg.shape[1] != dim):
        raise ValueError("feature widths differ")
    return points, refs, cent_pos, cent_neg


def _score_workspace(lib, points, refs, cent_pos, cent_neg):
    ws_bytes = lib.phm_score_workspace_bytes(points.shape[0], refs.shape[0], cent_pos.shape[0], cent_neg.shape[0], points.shape[1])
    ws = _workspace("score", ws_bytes)
    _last_score_ws[0] = ws
    return ws


def score_neighbors_cuda(points, refs, n_positive, cent_pos, cent_neg, k_neighbors=3):
    """score_cuda that also reports the rows behind each score, from the same device call (phm_score_neighbors).  Returns
    (knn, kmeans, combo float64[n] -- bit-identical to score_cuda --, ref_index int64[n, k] rows of `refs` of the k nearest references
    by ascending distance (ties: lower row first), ref_distance float64[n, k] their Euclidean distances, centroid_index int64[n, 2]
    rows of cent_pos / cent_neg of the nearest positive / negative centroid (-1 for an empty set), centroid_distance float64[n, 2]).
    A NaN query row reports index -1 and distance NaN."""
    lib = _lib.require_cuda()
    points, refs, cent_pos, cent_neg = _score_inputs(points, refs, cent_pos, cent_neg)
    n, dim = points.shape
    k = int(k_neighbors)
    knn, kmeans, combo = (torch.empty((n,), dtype=torch.float64, device="cuda") for _ in range(3))
    ref_index = torch.empty((n, max(k, 0)), dtype=torch.int64, device="cuda")
    ref_distance = torch.empty((n, max(k, 0)), dtype=torch.float64, device="cuda")
    centroid_index = torch.empty((n, 2), dtype=torch.int64, device="cuda")
    centroid_distance = torch.empty((n, 2), dtype=torch.float64, device="cuda")
    nb = _lib.Neighbors(ref_index.data_ptr(), ref_distance.data_ptr(), centroid_index.data_ptr(), centroid_distance.data_ptr())
    ws = _score_workspace(lib, points, refs, cent_pos, cent_neg)
    entry = lib.phm_score_counts_neighbors if points.dtype == torch.int32 else lib.phm_score_neighbors
    check(entry(ptr(points), n, dim, ptr(refs), refs.shape[0], int(n_positive),
                ptr(cent_pos), cent_pos.shape[0], ptr(cent_neg), cent_neg.shape[0], k,
                ptr(knn), ptr(kmeans), ptr(combo), ctypes.byref(nb), ptr(ws), ws.numel(), stream_ptr()))
    return knn, kmeans, combo, ref_index, ref_distance, centroid_index, centroid_distance


def count_score_cuda(seq, offsets, refs, n_positive, cent_pos, cent_neg, k_neighbors=3, out_counts=None, out=None):
    """The whole hot path in one call (k = 4): returns (counts int32[n, 256], knn, kmeans, combo float64[n]).
    Bit-identical to count_cuda followed by score_cuda on the counts; the histogram kernel prepares the scorer's operands."""
    lib = _lib.require_cuda()
    seq = _as_u8_cuda(seq)
    if not (isinstance(offsets, torch.Tensor) and offsets.is_cuda and offsets.dtype == torch.int64 and offsets.is_contiguous()):
        raise TypeError("offsets must be a contiguous CUDA int64 tensor")
    n = offsets.numel() - 1
    refs, cent_pos, cent_neg = (_check(t, name, torch.float64, 256) for t, name in
                                ((refs, "refs"), (cent_pos, "cent_pos"), (cent_neg, "cent_neg")))
    counts = _result(out_counts, (n, 256), torch.int32)
    knn, kmeans, combo = (_result(t, (n,), torch.float64) for t in (out if out is not None else (None, None, None)))
    ws_bytes = lib.phm_count_score_workspace_bytes(n, seq.numel(), refs.shape[0], cent_pos.shape[0], cent_neg.shape[0])
    ws = _workspace("count_score", ws_bytes)
    _last_score_ws[0] = ws
    check(lib.phm_count_score(ptr(seq), ptr(offsets), n, ptr(refs), refs.shape[0], int(n_positive), ptr(cent_pos), cent_pos.shape[0],
                              ptr(cent_neg), cent_neg.shape[0], int(k_neighbors), ptr(counts), ptr(knn), ptr(kmeans), ptr(combo),
                              ptr(ws), ws.numel(), stream_ptr()))
    return counts, knn, kmeans, combo


score_path_option = 0


def set_score_path(path):
    """'auto' (tensor cores when the shape allows; at width 136 for count rows only), 'exact' (exhaustive float64), 'tc' (tensor
    cores or error)."""
    global score_path_option
    score_path_option = {"auto": 0, "exact": 1, "tc": 2}[path]
    _lib.set_option("score_path", score_path_option)


def score_stats():
    """Diagnostics of the last tensor-core score_cuda call: rows re-scored by the exhaustive kernel, rows whose vote
    needed exact re-measurement, and (with _lib.set_option('score_stats', 1)) how much of the proven error interval the
    true ranking values use (must stay <= 1) and the largest ranking error in squared-distance units."""
    lib = _lib.require_cuda()
    ws = _last_score_ws[0]
    rows, err = ctypes.c_uint64(0), (ctypes.c_float * 4)()
    check(lib.phm_score_stats(ptr(ws), ctypes.byref(rows), err, stream_ptr()))
    return {"fallback_rows": int(rows.value), "max_bound_usage": float(err[0]), "max_rank_error": float(err[1]),
            "rows_remeasured": int(err[2]), "rows_listed": int(err[3])}


def fasta_scan_cuda(raw):
    """FASTA bytes on the device (contiguous CUDA uint8 tensor, 16-byte aligned) -> (seq uint8 [bases] end to end,
    offsets int64 [records + 1], header_pos int64 [records], odd_whitespace bool).  `seq` is padded to a multiple of 16
    bytes for phm_kmer_count.  One host synchronisation (the outputs are sized from the index pass).  When odd_whitespace is
    True (a control byte other than '\n' '\r' in the file: tab / VT / FF / 0x1C-0x1F are stripped by the reference at line
    ends only) use the host tokeniser.  The bytes of raw's storage past its end may hold anything."""
    lib = _lib.require_cuda()
    raw = _as_u8_cuda(raw)
    n = raw.numel()
    ws_bytes = lib.phm_fasta_workspace_bytes(n)
    ws = _workspace("fasta", ws_bytes)
    result = torch.empty((4,), dtype=torch.int64, device="cuda")
    check(lib.phm_fasta_index(ptr(raw), n, ptr(result), ptr(ws), ws_bytes, stream_ptr()))
    n_records, n_kept, odd, _ = [int(v) for v in result.cpu().tolist()]
    seq = torch.empty((max((n_kept + 15) // 16 * 16, 16),), dtype=torch.uint8, device="cuda")
    offsets = torch.empty((n_records + 1,), dtype=torch.int64, device="cuda")
    header_pos = torch.empty((max(n_records, 1),), dtype=torch.int64, device="cuda")
    check(lib.phm_fasta_extract(ptr(raw), n, ptr(result), ptr(seq), ptr(offsets), ptr(header_pos), n_records, ptr(ws), ws_bytes,
                                stream_ptr()))
    return seq, offsets, header_pos[:n_records], bool(odd)


def inflate_cuda(compressed, members, status=None):
    """phm_inflate: the members of a BGZF file (the table of fileIO.bgzf_members) decoded on the device.  compressed: CUDA uint8
    tensor of the file's bytes.  Returns a CUDA uint8 tensor of the decompressed file (members end to end) whose storage is padded
    to 16 bytes past the next multiple of 16, ready for fasta_scan_cuda.  status: optional CUDA int32 tensor [members] that
    receives each member's PHM_INFLATE_* status.  A member that fails to decode or whose CRC32 or length differs from its trailer
    raises _lib.PhamersDataError naming the lowest such member (one host synchronisation either way)."""
    import numpy as np
    from .fileIO import BGZF_MEMBER
    lib = _lib.require_cuda()
    if not (isinstance(compressed, torch.Tensor) and compressed.is_cuda and compressed.dtype == torch.uint8
            and compressed.is_contiguous()):
        raise TypeError("compressed must be a contiguous CUDA uint8 tensor")
    members = np.ascontiguousarray(members, dtype=BGZF_MEMBER)
    n = members.shape[0]
    total = int(members["out_offset"][-1]) + int(members["isize"][-1]) if n else 0
    out = torch.empty(((total + 15) // 16 * 16 + 16,), dtype=torch.uint8, device="cuda")
    status = _result(status, (n,), torch.int32) if status is not None else torch.empty((n,), dtype=torch.int32, device="cuda")
    ws = _workspace("inflate", lib.phm_inflate_workspace_bytes(n))
    check(lib.phm_inflate(ptr(compressed), compressed.numel(), members.ctypes.data_as(ctypes.c_void_p), n, ptr(out), total,
                          ptr(status), ptr(ws), ws.numel(), stream_ptr()))
    return out[:total]


def gunzip_cuda(compressed, member, stats=None):
    """phm_gunzip_index + phm_gunzip_extract: a single-member gzip file decoded on the device.  compressed: CUDA uint8 tensor of
    the file's bytes; member: fileIO.gzip_member of them (payload offset, payload end, CRC32, ISIZE).  Returns a CUDA uint8 tensor of
    the decompressed bytes whose storage is padded to 16 bytes past the next multiple of 16, ready for fasta_scan_cuda.  stats:
    optional dict that receives the index's diagnostics (chunks, rejected candidates, repair rounds, serial bytes, verified pieces,
    output bytes of the longest piece after the first).  A stream that
    zlib would refuse, or whose end, CRC32 or ISIZE differ from the trailer's, raises _lib.PhamersDataError; a device working set
    that does not fit raises torch.cuda.OutOfMemoryError.  Synchronises the host a few times (the chain of pieces is verified on
    the host between decode rounds)."""
    lib = _lib.require_cuda()
    if not (isinstance(compressed, torch.Tensor) and compressed.is_cuda and compressed.dtype == torch.uint8
            and compressed.is_contiguous()):
        raise TypeError("compressed must be a contiguous CUDA uint8 tensor")
    begin, end, crc, isize = (int(v) for v in member)
    if not 0 <= begin <= end <= compressed.numel():
        raise ValueError("the payload [%d, %d) is outside the %d bytes" % (begin, end, compressed.numel()))
    payload = compressed[begin:end]
    n = end - begin
    index_ws = torch.empty((lib.phm_gunzip_index_workspace_bytes(n),), dtype=torch.uint8, device="cuda")
    info = (ctypes.c_int64 * 7)()
    try:
        check(lib.phm_gunzip_index(ptr(payload), n, isize, info, ptr(index_ws), index_ws.numel(), stream_ptr()))
    finally:
        if stats is not None:
            stats.update(chunks=int(info[1]), rejected_candidates=int(info[2]), repair_rounds=int(info[3]),
                         serial_bytes=int(info[4]), pieces=int(info[5]), longest_later_piece_bytes=int(info[6]))
    total = int(info[0])
    out = torch.empty(((total + 15) // 16 * 16 + 16,), dtype=torch.uint8, device="cuda")
    ws = torch.empty((lib.phm_gunzip_extract_workspace_bytes(total),), dtype=torch.uint8, device="cuda")
    check(lib.phm_gunzip_extract(ptr(payload), n, crc, ptr(index_ws), index_ws.numel(), ptr(out), total, ptr(ws), ws.numel(),
                                 stream_ptr()))
    return out[:total]


def format_counts_csv_cuda(counts, id_bytes, id_offsets):
    """phm_counts_csv_layout + phm_counts_csv_format: the data rows of a feature CSV (fileIO.save_counts) written on the device.
    counts: CUDA int64 [n, F]; id_bytes: CUDA uint8, the ids end to end; id_offsets: CUDA int64 [n + 1] into id_bytes.  Returns a CUDA
    uint8 tensor of the text, row r being id_r + "," + ",".join(str(v) for v in counts[r]) + "\\n" ("id_r,\\n" when F = 0).  One host
    synchronisation (the text is sized from the layout pass)."""
    lib = _lib.require_cuda()
    counts = _check(counts, "counts", torch.int64)
    if counts.dim() != 2:
        raise ValueError("counts must be [rows, fields]")
    id_bytes = _check(id_bytes, "id_bytes", torch.uint8)
    id_offsets = _check(id_offsets, "id_offsets", torch.int64)
    n, f = counts.shape
    if id_offsets.shape != (n + 1,):
        raise ValueError("id_offsets must be [rows + 1]")
    row_offsets = torch.empty((n + 1,), dtype=torch.int64, device="cuda")
    ws_bytes = lib.phm_counts_csv_workspace_bytes(n)
    ws = _workspace("csv_format", ws_bytes)
    check(lib.phm_counts_csv_layout(ptr(counts), n, f, ptr(id_offsets), id_bytes.numel(), ptr(row_offsets), ptr(ws), ws_bytes,
                                    stream_ptr()))
    total = int(row_offsets[n].item())
    text = torch.empty((max(total, 1),), dtype=torch.uint8, device="cuda")
    check(lib.phm_counts_csv_format(ptr(counts), n, f, ptr(id_bytes), ptr(id_offsets), id_bytes.numel(), ptr(row_offsets), ptr(text),
                                    total, stream_ptr()))
    return text[:total]


def parse_feature_csv_cuda(text, result=None):
    """phm_feature_csv_index + phm_feature_csv_parse: a feature CSV on the device (contiguous CUDA uint8, 16-byte aligned, storage
    readable up to the next multiple of 16 bytes) -> (id byte ranges int64 [rows, 2] on the host, counts CUDA int64 [rows, F]), or None
    when the file is outside the device grammar (include/phamers_b200.h); the caller then parses it on the host.  result: optional
    CUDA int64 tensor [4] that receives the index block (rows, fields, PHM_CSV_* reason, line of the first decline).  One host
    synchronisation for the index, one for the id ranges."""
    import numpy as np
    lib = _lib.require_cuda()
    text = _as_u8_cuda(text)
    n = text.numel()
    ws_bytes = lib.phm_feature_csv_workspace_bytes(n)
    ws = _workspace("csv_parse", ws_bytes)
    result = _result(result, (4,), torch.int64)
    check(lib.phm_feature_csv_index(ptr(text), n, ptr(result), ptr(ws), ws_bytes, stream_ptr()))
    rows, fields, reason, _ = result.cpu().tolist()
    if reason != 0:
        return None
    counts = torch.empty((rows, fields), dtype=torch.int64, device="cuda")
    ranges = torch.empty((max(rows, 1), 2), dtype=torch.int64, device="cuda")
    check(lib.phm_feature_csv_parse(ptr(text), n, ptr(counts), ptr(ranges), rows, fields, ptr(ws), ws_bytes, stream_ptr()))
    return np.ascontiguousarray(ranges[:rows].cpu().numpy()), counts


def synth_contigs(seed, first_contig, n_contigs):
    """Synthetic metagenome shard (SURVEY.md 8(d) config 2) generated on the device.
    Returns (seq uint8[total], offsets int64[n+1])."""
    lib = _lib.require_cuda()
    lengths = torch.empty((n_contigs,), dtype=torch.int64, device="cuda")
    check(lib.phm_synth_lengths(ctypes.c_uint64(seed), int(first_contig), int(n_contigs), ptr(lengths), stream_ptr()))
    offsets = torch.zeros((n_contigs + 1,), dtype=torch.int64, device="cuda")
    torch.cumsum(lengths, 0, out=offsets[1:])
    total = int(offsets[-1].item())
    seq = torch.empty(((total + 15) // 16 * 16,), dtype=torch.uint8, device="cuda")
    check(lib.phm_synth_bases(ctypes.c_uint64(seed), int(first_contig), int(n_contigs), ptr(offsets), ptr(seq), stream_ptr()))
    return seq[:total], offsets


def last_kernel_ms(kernel="score_tc_kernel"):
    """Mean device time of the launches of a hot kernel ('kmer_hist_kernel', 'score_tc_kernel', 'score_decide_kernel') since the
    last call (after
    _lib.set_option('time_kernels', 1))."""
    ms = ctypes.c_float(0.0)
    check(_lib.require_cuda().phm_last_kernel_ms(kernel.encode(), ctypes.byref(ms)))
    return float(ms.value)

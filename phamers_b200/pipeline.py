"""
The whole hot path as one object: contigs in, PhaMers scores out.

    ContigScorer(positive, negative)          reference features (float64, normalised) -> device, centroids cached
      .score_device(seq, offsets)             device buffers -> (counts int32[n,256], scores float64[n]) on the device
      .score_host(seq, offsets)               HOST buffers (pinned recommended) -> numpy scores; copies included
      .score_fasta(path)                      FASTA file -> (ids, scores), the phamer.py flow without the files
      .score_windows_device(seq, offsets, w, s)   scores of overlapping windows along each record, on the device
      .score_windows_fasta(path, w, s)        FASTA file -> (ids, record index, spans, scores) of the windows
      .score_spans_device(seq, offsets, spans)    scores (and neighbours) of arbitrary (record, start, end) spans, on the device
      .score_spans_fasta(path, ids, spans)    FASTA file + contig-named spans (a BED file) -> their scores on the host

Stage by stage this is kmer.count_file -> kmer.normalize_counts -> phamer_scorer.score_points('combo')
(reference scripts/phamer.py:131,139,194), with the k-mer length fixed at the width of the reference features.

ContigScorer(..., canonical=True) scores canonical 4-mers (each k-mer folded with its reverse complement, 136 bins), so a contig
and its reverse complement get the same score: references are 136 wide, contigs are counted with PHM_COUNT_CANONICAL and scored
from the counts.

ContigScorer(..., kmer_length=5[, canonical=True]) takes 5-mer reference rows (1024 or 512 wide: the shipped tables are 4-mer, so
the caller passes its own); score_device / score_host / score_fasta count the contigs at k = 5 and score the counts on the
tensor-core road at that width.  Windows and spans are scored from feature rows on the exhaustive kernel, as before.
"""
import numpy as np
import torch

from . import _lib, ops, references


def match_records(names, ids, tokens):
    """Record index of every contig name: first among `ids` (the score file's ids, fileIO.get_id of each title), then, when no id
    matches, among `tokens` (the titles' first whitespace tokens).  A name that matches no record, or more than one, is a ValueError
    naming it."""
    def index(keys):
        table = {}
        for r, key in enumerate(keys):
            if key is not None:
                table.setdefault(str(key), []).append(r)
        return table
    by_id, by_token = index(ids), index(tokens)
    out = np.empty((len(names),), dtype=np.int64)
    for i, name in enumerate(names):
        hits = by_id.get(str(name)) or by_token.get(str(name))
        if not hits:
            raise ValueError("contig %r names no record of the FASTA file" % (name,))
        if len(hits) > 1:
            raise ValueError("contig %r names %d records of the FASTA file" % (name, len(hits)))
        out[i] = hits[0]
    return out


def fasta_spans(path, ids, spans, lines=None):
    """A FASTA file and contig-named spans (ids [n], spans [n, 2] start, end) -> (sequence bytes and offsets on the device, the span
    table int64[n, 3] (record, start, end) on the device).  Names are matched by match_records; coordinates outside their record are
    a ValueError naming lines[i] (where the span came from) when given."""
    from . import fileIO
    tokens, d_seq, d_off = fileIO.read_fasta_arrays_cuda(path)
    records = match_records(ids, [fileIO.get_id(t) for t in tokens], tokens)
    spans = np.asarray(spans, dtype=np.int64).reshape(-1, 2)
    lengths = np.diff(d_off.cpu().numpy())
    for i in np.flatnonzero((spans[:, 0] < 0) | (spans[:, 1] < spans[:, 0]) | (spans[:, 1] > lengths[records])):
        where = lines[i] if lines is not None else "span %d" % i
        raise ValueError("%s: [%d, %d) is not a range inside %s (%d bases)" % (where, spans[i, 0], spans[i, 1], ids[i], lengths[records[i]]))
    table = np.ascontiguousarray(np.concatenate((records[:, None], spans), axis=1))
    return d_seq, d_off, torch.from_numpy(table).cuda()


class ContigScorer(object):
    def __init__(self, positive=None, negative=None, k_clusters=86, k_neighbors=3, kmer_length=4, centroids=None,
                 equalize=True, canonical=False):
        _lib.require_cuda()
        if positive is None or negative is None:
            positive, negative = references.load_reference_features(equalize=equalize, canonical=canonical)
        positive = np.ascontiguousarray(positive, dtype=np.float64)
        negative = np.ascontiguousarray(negative, dtype=np.float64)
        width = ops.num_bins(kmer_length, canonical)
        if positive.shape[1] != width or negative.shape[1] != width:
            raise ValueError("reference features are %d wide, k = %d%s needs %d"
                             % (positive.shape[1], kmer_length, " canonical" if canonical else "", width))
        self.canonical = canonical
        if centroids is None:
            centroids = references.reference_centroids(positive, negative, k_clusters)
        self.kmer_length = kmer_length
        self.k_neighbors = k_neighbors
        self.n_positive = positive.shape[0]
        self.refs = torch.from_numpy(np.vstack((positive, negative))).cuda()
        self.cent_pos = torch.from_numpy(np.ascontiguousarray(centroids[0], dtype=np.float64)).cuda()
        self.cent_neg = torch.from_numpy(np.ascontiguousarray(centroids[1], dtype=np.float64)).cuda()
        self._staging = None
        self._host_out = None
        self._copy_stream = None
        self._chunk_counts = None

    # -- device resident --------------------------------------------------------------------------------
    def score_device(self, seq, offsets, method="combo", return_counts=True):
        # one library call: the histogram kernel also emits the scorer's query operands, the scorer forms count / row total
        # wherever it needs an exact feature; the float64 feature matrix is never written
        counts, knn, kmeans, combo = self._count_score(seq, offsets)
        return counts, {"knn": knn, "kmeans": kmeans, "combo": combo}[method]

    def _count_score(self, seq, offsets, out_counts=None, out=None):
        if not self.canonical and self.kmer_length == 4:
            return ops.count_score_cuda(seq, offsets, self.refs, self.n_positive, self.cent_pos, self.cent_neg, self.k_neighbors,
                                        out_counts=out_counts, out=out)
        # canonical or 5-mer counts, then phm_score_counts on them (the fused count + score call emits plain 256-wide operands only)
        counts, _ = ops.count_cuda(seq, offsets, self.kmer_length, canonical=self.canonical, out_counts=out_counts)
        return (counts,) + ops.score_cuda(counts, self.refs, self.n_positive, self.cent_pos, self.cent_neg, self.k_neighbors, out=out)

    # -- host buffers -----------------------------------------------------------------------------------
    HOST_CHUNKS = 8                    # upload / compute pipeline depth of score_host
    HOST_CHUNK_MIN_BASES = 1 << 22     # ... and the least bases worth a range of its own

    def score_host(self, seq, offsets, method="combo"):
        """seq: uint8 host tensor / ndarray with all contigs end to end (pinned memory makes the copies asynchronous), offsets:
        int64[n+1].  The contigs are cut into HOST_CHUNKS ranges of about equal bases; range i + 1 is copied to the device on a
        copy stream while range i is counted and scored, and the scores come back in one copy at the end.  The host -> device
        copy (16 GB per million contigs against ~9 ms of compute) is what bounds this call: see DESIGN.md section 7."""
        seq_t = seq if isinstance(seq, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(seq))
        off_t = offsets if isinstance(offsets, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(offsets, dtype=np.int64))
        n = off_t.numel() - 1
        if n <= 0:
            return np.zeros((0,), dtype=np.float64)
        host_off = off_t.numpy()
        total = int(host_off[-1] - host_off[0])
        n_chunks = max(1, min(self.HOST_CHUNKS, n, total // self.HOST_CHUNK_MIN_BASES + 1))
        targets = host_off[0] + (total * np.arange(1, n_chunks, dtype=np.float64) / n_chunks)
        cuts = np.unique(np.concatenate(([0], np.clip(np.searchsorted(host_off, targets, side="left"), 0, n), [n])))
        padded = (total + 15) // 16 * 16 + 32 * len(cuts)
        if self._staging is None or self._staging.numel() < padded:
            self._staging = torch.empty((padded,), dtype=torch.uint8, device="cuda")
        if self._host_out is None or self._host_out.numel() < n:
            self._host_out = torch.empty((n,), dtype=torch.float64, pin_memory=True)             # pinned once, reused
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream()
        main = torch.cuda.current_stream()
        d_off = off_t.to("cuda", non_blocking=True)
        scores = torch.empty((n,), dtype=torch.float64, device="cuda")
        widest = int(np.max(np.diff(cuts)))
        if self._chunk_counts is None or self._chunk_counts.shape[0] < widest:
            self._chunk_counts = torch.empty((widest, self.refs.shape[1]), dtype=torch.int32, device="cuda")
        self._copy_stream.wait_stream(main)                                  # the staging buffer may still be read by an earlier call
        uploads, place = [], 0
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            b0, b1 = int(host_off[lo]), int(host_off[hi])
            dst = self._staging[place:place + (b1 - b0)]
            with torch.cuda.stream(self._copy_stream):
                dst.copy_(seq_t[b0:b1], non_blocking=True)
                done = torch.cuda.Event()
                done.record(self._copy_stream)
            uploads.append((int(lo), int(hi), b0, dst, done))
            place += (b1 - b0 + 15) // 16 * 16 + 16                          # every range starts 16-byte aligned, padding readable
        key = {"knn": 0, "kmeans": 1, "combo": 2}[method]
        for lo, hi, b0, dst, done in uploads:
            main.wait_event(done)
            part = [torch.empty((hi - lo,), dtype=torch.float64, device="cuda") if i != key else scores[lo:hi] for i in range(3)]
            self._count_score(dst, d_off[lo:hi + 1] - b0, out_counts=self._chunk_counts[:hi - lo], out=tuple(part))
        out = self._host_out[:n]
        out.copy_(scores, non_blocking=True)
        main.synchronize()
        return out.numpy().copy()

    # -- sliding windows ---------------------------------------------------------------------------------
    WINDOW_SLICE = 1 << 20             # windows counted and scored per library call: bounds the count rows (1 GB at 256 bins)

    def score_windows_device(self, seq, offsets, window, step, method="combo"):
        """Scores of overlapping windows along every record (phm_window_offsets, phm_kmer_count_windows, then the scorer on the
        count rows).  Returns, on the device, (window offsets int64[n_records + 1], spans int64[n_windows, 2] -- start, end relative
        to the record --, scores float64[n_windows]).  Windows are counted and scored WINDOW_SLICE at a time.  Count rows go to the
        scorer as counts where the count road takes them (k_neighbors in {1, 3, 5}); other shapes are scored from float64 feature rows
        normalised by the same call.  A window with no countable k-mer scores NaN."""
        key = {"knn": 0, "kmeans": 1, "combo": 2}[method]
        wo = ops.window_offsets_cuda(offsets, window, step)
        total = int(wo[-1].item())
        spans = torch.empty((total, 2), dtype=torch.int64, device="cuda")
        scores = torch.empty((total,), dtype=torch.float64, device="cuda")
        from_counts = (self.k_neighbors in (1, 3, 5) and self.refs.shape[1] in (256, 136)
                       and self.cent_pos.shape[0] > 0 and self.cent_neg.shape[0] > 0)
        for first in range(0, total, self.WINDOW_SLICE):
            n = min(self.WINDOW_SLICE, total - first)
            counts, freq, sp = ops.count_windows_cuda(seq, offsets, wo, window, step, self.kmer_length, first=first, n=n,
                                                      canonical=self.canonical, counts=from_counts, freq=not from_counts, spans=True)
            spans[first:first + n] = sp
            out = tuple(scores[first:first + n] if i == key else torch.empty((n,), dtype=torch.float64, device="cuda")
                        for i in range(3))
            ops.score_cuda(counts if from_counts else freq, self.refs, self.n_positive, self.cent_pos, self.cent_neg,
                           self.k_neighbors, out=out)
        return wo, spans, scores

    def score_windows_fasta(self, path, window, step, length_requirement=0, method="combo"):
        """score_windows_device over the records of a FASTA file.  Returns on the host (ids [n_windows] -- the id of each window's
        record --, record_index int64[n_windows] -- its position in the file --, spans int64[n_windows, 2], scores float64[n_windows]),
        with the windows of records shorter than length_requirement left out."""
        from . import fileIO
        headers, d_seq, d_off = fileIO.read_fasta_arrays_cuda(path)
        ids = np.array([fileIO.get_id(h) for h in headers])
        if len(ids) == 0:
            return ids, np.zeros((0,), dtype=np.int64), np.zeros((0, 2), dtype=np.int64), np.zeros((0,), dtype=np.float64)
        wo, spans, scores = self.score_windows_device(d_seq, d_off, window, step, method=method)
        wo, spans, scores = wo.cpu().numpy(), spans.cpu().numpy(), scores.cpu().numpy()
        record = np.repeat(np.arange(len(ids), dtype=np.int64), np.diff(wo))
        keep = (np.diff(d_off.cpu().numpy()) >= length_requirement)[record]
        return ids[record[keep]], record[keep], spans[keep], scores[keep]

    # -- spans ------------------------------------------------------------------------------------------
    SPAN_SLICE = 1 << 20               # spans counted and scored per library call, as WINDOW_SLICE

    def score_spans_device(self, seq, offsets, spans, method="combo", neighbors=False):
        """Scores of arbitrary spans of the records (phm_kmer_count_spans, then the scorer on the count rows).  spans: int64 CUDA tensor
        [n, 3] of (record, start, end), 0-based half-open in the record, any order.  A span scores exactly as its bases would as a
        record of their own (score_fasta); one without a countable k-mer scores NaN.  Spans are counted and scored SPAN_SLICE at a
        time, count rows on the count road where it takes them (k_neighbors in {1, 3, 5}), other shapes from feature rows normalised
        by the same call.  Returns scores float64[n] on the device; with neighbors=True the tuple (scores, ref_index int64[n, k],
        ref_distance, centroid_index int64[n, 2], centroid_distance) of ops.score_neighbors_cuda for the same rows."""
        key = {"knn": 0, "kmeans": 1, "combo": 2}[method]
        n_spans = spans.shape[0]
        from_counts = (self.k_neighbors in (1, 3, 5) and self.refs.shape[1] in (256, 136)
                       and self.cent_pos.shape[0] > 0 and self.cent_neg.shape[0] > 0)
        parts = []
        for first in range(0, n_spans, self.SPAN_SLICE):
            part = spans[first:first + self.SPAN_SLICE]
            counts, freq = ops.count_spans_cuda(seq, offsets, part, self.kmer_length, canonical=self.canonical, counts=from_counts,
                                                freq=not from_counts)
            args = (counts if from_counts else freq, self.refs, self.n_positive, self.cent_pos, self.cent_neg, self.k_neighbors)
            out = ops.score_neighbors_cuda(*args) if neighbors else ops.score_cuda(*args)
            parts.append((out[key],) + tuple(out[3:]))
        if not parts:
            parts = [(torch.empty((0,), dtype=torch.float64, device="cuda"), torch.empty((0, self.k_neighbors), dtype=torch.int64, device="cuda"),
                      torch.empty((0, self.k_neighbors), dtype=torch.float64, device="cuda"),
                      torch.empty((0, 2), dtype=torch.int64, device="cuda"), torch.empty((0, 2), dtype=torch.float64, device="cuda"))]
        joined = tuple(torch.cat(col) for col in zip(*parts))
        return joined if neighbors else joined[0]

    def score_spans_fasta(self, path, ids, spans, method="combo", neighbors=False, lines=None):
        """score_spans_device over the records of a FASTA file, spans named by contig: ids [n] names, spans int64[n, 2] (start, end).
        A name is looked up among the score file's ids (fileIO.get_id of each title) first and, when none has it, among the titles'
        first tokens (what BED files of other tools carry); a name that matches no record or several is a ValueError naming it, and
        so are coordinates outside their record (naming lines[i], the span's source, when given).  Returns on the host what
        score_spans_device returns, as numpy arrays."""
        d_seq, d_off, table = fasta_spans(path, ids, spans, lines)
        out = self.score_spans_device(d_seq, d_off, table, method=method, neighbors=neighbors)
        return tuple(t.cpu().numpy() for t in out) if neighbors else out.cpu().numpy()

    def score_fasta(self, path, length_requirement=0, method="combo"):
        from . import fileIO
        headers, d_seq, d_off = fileIO.read_fasta_arrays_cuda(path)      # records are found on the device; the bases stay there
        ids = np.array([fileIO.get_id(h) for h in headers])
        if len(ids) == 0:
            return ids, np.zeros((0,), dtype=np.float64)
        _, d_scores = self.score_device(d_seq, d_off, method=method, return_counts=False)
        scores = d_scores.cpu().numpy()
        if length_requirement:
            keep = np.diff(d_off.cpu().numpy()) >= length_requirement    # scripts/phamer.py:154
            ids, scores = ids[keep], scores[keep]
        return ids, scores

/*
 * phamers_b200 -- C-ABI of the B200-native PhaMers hot path (k-mer count -> normalise -> score).
 *
 * The reference (jondeaton/PhaMers) is pure Python and has no FFI of its own; the boundary it exposes
 * for this path is the module-level API of scripts/kmer.py and scripts/phamer.py.  The entry points
 * below are what a ctypes binding inside those two modules calls (see INTEGRATION.md); each one cites
 * the reference lines it replaces (paths relative to the reference checkout).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only.  Every `d_*` pointer is a DEVICE pointer on the
 *     current CUDA device; `h_*` marks the few HOST pointers (small result blocks).
 *   - All launches go to `stream` (a cudaStream_t / CUstream passed as void*; NULL = default stream).
 *     Entry points never allocate; scratch memory is caller-owned (`d_workspace`, sized by the matching
 *     *_workspace_bytes function) and they do not synchronise unless their comment says so.
 *   - Concurrency: calls that use DIFFERENT workspaces may run concurrently on different streams, threads
 *     and devices.  A workspace holds live kernel state (work counters, candidate lists), so two calls
 *     must never share one while either is in flight.  The tuning options of phm_set_option and the
 *     timing hooks (phm_last_kernel_ms, phm_kernel_launches) are PROCESS-WIDE and not synchronised: set
 *     them while no call is running.
 *   - Sequence buffers (`d_seq`, `d_raw`) are read with 128-bit loads: they must be 16-byte aligned and
 *     the allocation must be READABLE up to the next multiple of 16 bytes past the last base (the
 *     content of that padding does not matter).
 *   - Return value: 0 = ok, negative = error (PHM_E_*); phm_last_error() gives the message of the
 *     most recent failure on the calling thread.
 *   - Bin order everywhere is the reference's: symbols 'ATGC' (A=0 T=1 G=2 C=3), first base most
 *     significant (scripts/kmer.py:28,44-50,183-196).  Only those four upper-case bytes are symbols;
 *     any other byte voids every window it touches.
 */
#ifndef PHAMERS_B200_H
#define PHAMERS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PHM_VERSION 100            /* 0.1.0 */

#define PHM_OK             0
#define PHM_E_ARG         -1       /* bad argument (k out of range, null pointer, misaligned buffer) */
#define PHM_E_CUDA        -2       /* a CUDA runtime call failed; see phm_last_error() */
#define PHM_E_WORKSPACE   -3       /* workspace too small */
#define PHM_E_UNSUPPORTED -4       /* not an sm_100 device / option not built */

/* flags for phm_kmer_count* */
#define PHM_COUNT_CANONICAL  1u    /* fold reverse complements: out bins = 136 / 512 / 2080 for k = 4 / 5 / 6 */
#define PHM_COUNT_NAIVE      2u    /* use the simple (slow) cross-check kernel */

typedef struct phm_caps {
    int32_t device;                /* CUDA device ordinal */
    int32_t sm_major, sm_minor;    /* 10, 0 on B200 */
    int32_t sm_count;              /* 148 on B200 */
    int32_t max_smem_optin;        /* bytes of shared memory per CTA (227 KB on B200) */
    int64_t hbm_bytes;             /* total device memory */
} phm_caps;

int          phm_version(void);
const char  *phm_last_error(void);
int          phm_device_caps(phm_caps *out);

/* Number of output bins for k (4^k), or for the canonical fold (136 / 512 / 2080 ...). */
int64_t      phm_num_bins(int k, uint32_t flags);

/* ---------------------------------------------------------------------------------------------
 * K1  sequence pack.  Replaces kmer.sequence_to_integers (scripts/kmer.py:183-196): ASCII bases ->
 *     2-bit codes in reference order (A=0 T=1 G=2 C=3), 16 bases per uint32 with the FIRST base in the
 *     top two bits (base i of a word in bits 31-2i:30-2i, so the bin of the k-mer starting at base i
 *     is the plain bit field (word >> (32-2i-2k)) & (4^k-1)), plus one validity bit per base, 32 bases
 *     per uint32, first base in the top bit (bit 31-i = base i is one of ATGC; codes of other bytes are 0).
 *     d_seq must be 16-byte aligned.  d_codes holds ceil(n_bases/16) words, d_valid ceil(n_bases/32).
 * ------------------------------------------------------------------------------------------- */
int phm_pack_fasta(const uint8_t *d_seq, int64_t n_bases, uint32_t *d_codes, uint32_t *d_valid, void *stream);

/* ---------------------------------------------------------------------------------------------
 * K2+K3  k-mer histogram with fused (optional canonical) fold and normalisation.
 *     Replaces the loop of kmer.count_string (scripts/kmer.py:42-50) over every record of
 *     kmer.count_file (scripts/kmer.py:137-139) and kmer.normalize_counts (scripts/kmer.py:209-221).
 *
 *     d_seq      ASCII bases of all contigs laid end to end (record text with line breaks already
 *                removed, i.e. what str(record.seq) is in the reference); 16-byte aligned.
 *     d_offsets  int64[n_contigs + 1]; contig i = d_seq[d_offsets[i] .. d_offsets[i+1]).
 *     k          1..6.
 *     d_counts   uint32[n_contigs * bins]          (may be NULL)  -- bit-exact with the reference.
 *     d_freq     float64[n_contigs * bins]         (may be NULL)  -- counts / row sum, IEEE division
 *                exactly as numpy does it; an all-zero row gives NaN like kmer.py:219-220.
 *     d_workspace / workspace_bytes  scratch from phm_kmer_count_workspace_bytes(n_contigs, n_bases, ...).  Its size grows with
 *                n_bases because it holds the list of work items of records that are cut into tiles (131 072 bases and more are
 *                counted by many warps and merged).  A workspace sized for fewer bases than the offsets describe is legal: such
 *                records are then counted whole by one warp each.
 * ------------------------------------------------------------------------------------------- */
size_t phm_kmer_count_workspace_bytes(int64_t n_contigs, int64_t n_bases, int k, uint32_t flags);
int phm_kmer_count(const uint8_t *d_seq, const int64_t *d_offsets, int64_t n_contigs, int k, uint32_t flags,
                   uint32_t *d_counts, double *d_freq,
                   void *d_workspace, size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Sliding windows: the same histogram over overlapping windows of every record, to find where in a long sequence (a prophage in a
 * bacterial contig, a chimeric assembly) the phage-like part lies.  Coordinates are 0-based, half-open, relative to the record.
 * For a record of length L, window w >= 1 and step s >= 1: one window [0, L) when L <= w (L = 0 included); otherwise [j s, j s + w)
 * for j = 0, 1, ... while j s + w <= L, then [L - w, L) when the last of those ends before L -- 1 + ceil((L - w) / s) windows, each
 * w long, numbered in ascending start order, records in order.  A window's counts are exactly phm_kmer_count's counts of the range
 * (k-mers wholly inside it; bytes that are not symbols void the k-mers they touch); a window with none gets a NaN feature row.
 *
 *   phm_window_offsets      d_window_offsets int64[n_records + 1]: [0] = 0, record r owns windows [wo[r], wo[r + 1]).
 *   phm_kmer_count_windows  counts the windows [first_window, first_window + n_windows) into rows 0 .. n_windows - 1 of d_counts /
 *                           d_freq (phm_kmer_count's outputs and flags; PHM_COUNT_NAIVE is not accepted), and writes each window's
 *                           (start, end) relative to its record to d_spans[2 i], [2 i + 1] (may be NULL).  The workspace
 *                           (phm_kmer_count_windows_workspace_bytes) holds one 32-byte work item per window, or w / 65 536 of them
 *                           for windows of 131 072 bases and more (counted in tiles); a smaller one is PHM_E_WORKSPACE.  Argument
 *                           errors are PHM_E_ARG; the slice is checked against wo[n_records], which the call reads from the device
 *                           (it synchronises `stream` once).  Score the rows with phm_score_counts / phm_score.
 * ------------------------------------------------------------------------------------------- */
int phm_window_offsets(const int64_t *d_offsets, int64_t n_records, int64_t window, int64_t step, int64_t *d_window_offsets,
                       void *stream);
size_t phm_kmer_count_windows_workspace_bytes(int64_t n_windows, int64_t window, int k, uint32_t flags);
int phm_kmer_count_windows(const uint8_t *d_seq, const int64_t *d_offsets, int64_t n_records, const int64_t *d_window_offsets,
                           int64_t window, int64_t step, int64_t first_window, int64_t n_windows, int k, uint32_t flags,
                           uint32_t *d_counts, double *d_freq, int64_t *d_spans,
                           void *d_workspace, size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Spans: the same histogram over arbitrary pieces of the records -- a phage-like region, a gene, the intervals of a BED file.
 * d_spans is int64[n_spans * 3]: (record, start, end) per span, 0-based, half-open, relative to the record, in any order; spans may
 * overlap, repeat, be empty or be shorter than k.  Row i of d_counts / d_freq holds span i: exactly phm_kmer_count's counts of
 * d_seq[off[record] + start, off[record] + end) taken as a record of its own (plain or PHM_COUNT_CANONICAL, the only flag accepted);
 * a span with no countable k-mer gets a NaN feature row.  The workspace (phm_kmer_count_spans_workspace_bytes, n_span_bases = the
 * summed span length) holds one 32-byte work item per span plus the tiles of spans of 131 072 bases and more.
 * Argument errors (k, flags, sizes, null or misaligned pointers) are PHM_E_ARG and a workspace without one item per span is
 * PHM_E_WORKSPACE, both before the device is touched.  The call then validates every span on the device and synchronises `stream`
 * once to read the result: a span whose record is not in [0, n_records), whose start is < 0, whose end is < its start or past its
 * record's end is PHM_E_ARG naming the lowest such index and its fields, and a list that does not fit the workspace is
 * PHM_E_WORKSPACE; in both cases no output row has been written.  Score the rows with phm_score_counts / phm_score.
 * ------------------------------------------------------------------------------------------- */
size_t phm_kmer_count_spans_workspace_bytes(int64_t n_spans, int64_t n_span_bases, int k, uint32_t flags);
int phm_kmer_count_spans(const uint8_t *d_seq, const int64_t *d_offsets, int64_t n_records,
                         const int64_t *d_spans, int64_t n_spans, int k, uint32_t flags,
                         uint32_t *d_counts, double *d_freq, void *d_workspace, size_t workspace_bytes, void *stream);

/* Same histogram from the packed form produced by phm_pack_fasta (multi-k passes over one pack). */
int phm_kmer_count_packed(const uint32_t *d_codes, const uint32_t *d_valid, const int64_t *d_offsets,
                          int64_t n_contigs, int k, uint32_t flags, uint32_t *d_counts, double *d_freq,
                          void *d_workspace, size_t workspace_bytes, void *stream);

/* Canonical fold of rows that already exist: float64 d_rows[n_rows * 4^k] -> d_out[n_rows * phm_num_bins(k, PHM_COUNT_CANONICAL)],
 * k = 1..6, with the definition and bin order of phm_kmer_count(..., PHM_COUNT_CANONICAL): out[c] = row[y] + row[rc(y)] for the c-th
 * smallest y with y <= rc(y) (row[y] alone when y = rc(y)).  One add per bin pair, so integer-valued rows below 2^53 fold exactly.
 * Needs no workspace; d_rows and d_out must not overlap.  Folding commutes with summing rows, and a row's total does not change, so
 * fold-then-normalise equals normalising canonical counts. */
int phm_canonical_fold(const double *d_rows, int64_t n_rows, int k, double *d_out, void *stream);

/* kmer.normalize_counts on its own (scripts/kmer.py:209-221) for counts that are already on the device. */
int phm_normalize_counts(const uint32_t *d_counts, int64_t n_rows, int64_t bins, double *d_freq, void *stream);
/* The same for rows that are not exact 32-bit counts (the summed genome counts of kmer.count_directory, already-float features):
 * float64 row / row sum.  Equals numpy's result for integer-valued rows with sums below 2^53; otherwise the row sum may differ
 * from numpy's pairwise sum in the last bit. */
int phm_normalize_rows(const double *d_rows, int64_t n_rows, int64_t bins, double *d_out, void *stream);

/* ---------------------------------------------------------------------------------------------
 * K4+K5  scoring.  Replaces phamer_scorer.knn_score_points / kmeans_score_points / combo_score_points
 *     (scripts/phamer.py:240-256,268-273,303-313), i.e. learning.knn (scripts/learning.py:118-128),
 *     learning.closest_to (:59-66) and phamer_scorer.proximity_metric (scripts/phamer.py:198-210).
 *     Clustering of the reference sets (learning.kmeans, :131-146) is reference-only preprocessing and
 *     stays on the host: the caller passes the centroids.
 *
 *     d_points        float64[n_points * dim]   query features (rows of kmer.normalize_counts)
 *     d_refs          float64[n_refs * dim]     positive rows first, then negative (phamer.py:186)
 *     n_positive      number of leading rows of d_refs labelled 1 (phamer.py:187)
 *     d_cent_pos/neg  float64[n_cent_* * dim]   centroids of the positive / negative clusters
 *     k_neighbors     odd, 1..15 (reference default 3, phamer.py:79)
 *     d_knn           float64[n_points]  +1 / -1 vote                    (may be NULL)
 *     d_kmeans        float64[n_points]  tanh((e_neg-e_pos)/(e_pos+e_neg))  (may be NULL)
 *     d_combo         float64[n_points]  knn + kmeans                     (may be NULL)
 *     A query row holding NaN (zero-count contig) gets NaN in all three outputs.
 *
 *     Two device paths, same results: for dim = 256, 136, 1024 or 512 and k_neighbors in {1, 3, 5} the (query x reference)
 *     contraction runs on
 *     the tcgen05 tensor cores (FP16 operands, FP32 accumulation) together with a proven per-pair error interval; the few
 *     references / centroids whose interval can reach the k nearest are kept per query and decided exactly in float64.
 *     Rows whose candidate buffer overflows (and every other shape) go through the exhaustive float64 kernel.
 *     See DESIGN.md section 5 for the error bound.
 *     dim = 136 is the width of canonical 4-mer features (phm_canonical_fold, PHM_COUNT_CANONICAL at k = 4): their rows fill the
 *     first 136 columns of the 256-wide FP16 operands and the rest is zero, under the same error bound.  At dim = 136 count rows
 *     (phm_score_counts) take the tensor cores; float64 feature rows keep the exhaustive kernel unless option "score_path" = 2,
 *     because the two roads may order exact distance ties differently and phm_score's answers at 136 stay what they were.
 *     dim = 1024 and 512 are the widths of plain and canonical 5-mer features: their FP16 operands are that wide (the workspace
 *     grows with them, phm_score_workspace_bytes takes dim).  As at 136, count rows take the tensor cores and float64 feature rows
 *     keep the exhaustive kernel unless option "score_path" = 2.
 * ------------------------------------------------------------------------------------------- */
size_t phm_score_workspace_bytes(int64_t n_points, int64_t n_refs, int64_t n_cent_pos, int64_t n_cent_neg, int dim);
int phm_score(const double *d_points, int64_t n_points, int dim,
              const double *d_refs, int64_t n_refs, int64_t n_positive,
              const double *d_cent_pos, int64_t n_cent_pos, const double *d_cent_neg, int64_t n_cent_neg,
              int k_neighbors, double *d_knn, double *d_kmeans, double *d_combo,
              void *d_workspace, size_t workspace_bytes, void *stream);

/* Stages 2 + 3 fused: same as phm_score, but the queries are the raw uint32 count rows of phm_kmer_count (d_counts[n_points * dim]);
 * every kernel forms feature = count / row total in float64 on the fly, exactly as kmer.normalize_counts would
 * (scripts/kmer.py:209-221, scripts/phamer.py:139), so the float64 feature matrix never exists in memory.  Needs the
 * tensor-core shape (dim = 256 or 136 -- plain or canonical 4-mer counts --, 1024 or 512 -- plain or canonical 5-mer counts --,
 * k_neighbors in {1, 3, 5}, both centroid sets),
 * PHM_E_UNSUPPORTED otherwise. */
int phm_score_counts(const uint32_t *d_counts, int64_t n_points, int dim,
                     const double *d_refs, int64_t n_refs, int64_t n_positive,
                     const double *d_cent_pos, int64_t n_cent_pos, const double *d_cent_neg, int64_t n_cent_neg,
                     int k_neighbors, double *d_knn, double *d_kmeans, double *d_combo,
                     void *d_workspace, size_t workspace_bytes, void *stream);

/* Neighbour report: the rows that decided each score, written by the same call that writes the scores.
 *     For query row i, with k = k_neighbors and references in d_refs order (positives first):
 *     d_ref_index[i*k .. i*k+k-1]       rows of d_refs of the k nearest references, ascending float64 Euclidean distance, ties to
 *                                       the lower row first (the references whose labels cast the vote)
 *     d_ref_distance[i*k .. i*k+k-1]    their distances: sqrt of the float64 direct-difference sum of squares (the arithmetic of
 *                                       phm_distances, not the |a|^2 + |b|^2 - 2ab expansion)
 *     d_centroid_index[2i], [2i+1]      row of d_cent_pos of the nearest positive centroid, row of d_cent_neg of the nearest negative
 *                                       one (first on ties, like np.argmin; -1 when that centroid set is empty).  With centroids from
 *                                       k-means, the row is the cluster label.
 *     d_centroid_distance[2i], [2i+1]   their distances: the e_pos, e_neg of tanh((e_neg - e_pos)/(e_pos + e_neg))
 *     A NaN query row reports index -1 and distance NaN in every slot.  Every member may be NULL. */
typedef struct phm_neighbors {
    int64_t *d_ref_index;          /* int64  [n_points * k_neighbors]  (may be NULL) */
    double  *d_ref_distance;       /* float64[n_points * k_neighbors]  (may be NULL) */
    int64_t *d_centroid_index;     /* int64  [n_points * 2]  nearest positive, nearest negative (may be NULL) */
    double  *d_centroid_distance;  /* float64[n_points * 2]  (may be NULL) */
} phm_neighbors;

/* phm_score / phm_score_counts that also fill `nb` (same arguments, same workspace size from phm_score_workspace_bytes).  The
 * scores are bit-identical to those of phm_score / phm_score_counts on the same inputs, and consistent with the report: the labels
 * of the reported references give the vote, tanh((cd[1] - cd[0]) / (cd[0] + cd[1])) is the kmeans score.  On the tensor-core path
 * every live row has its candidate band re-measured exactly (the vote alone may be settled by the error intervals; the order of the
 * k nearest is not), which costs time; on the exhaustive path (other widths, k outside {1, 3, 5}) the k references are selected by
 * the norm expansion and then re-measured, so at a near tie (gap below the expansion's rounding) that path may report the other
 * member of the tie.  nb = NULL, or all members NULL: exactly phm_score / phm_score_counts. */
int phm_score_neighbors(const double *d_points, int64_t n_points, int dim,
                        const double *d_refs, int64_t n_refs, int64_t n_positive,
                        const double *d_cent_pos, int64_t n_cent_pos, const double *d_cent_neg, int64_t n_cent_neg,
                        int k_neighbors, double *d_knn, double *d_kmeans, double *d_combo, const phm_neighbors *nb,
                        void *d_workspace, size_t workspace_bytes, void *stream);
int phm_score_counts_neighbors(const uint32_t *d_counts, int64_t n_points, int dim,
                               const double *d_refs, int64_t n_refs, int64_t n_positive,
                               const double *d_cent_pos, int64_t n_cent_pos, const double *d_cent_neg, int64_t n_cent_neg,
                               int k_neighbors, double *d_knn, double *d_kmeans, double *d_combo, const phm_neighbors *nb,
                               void *d_workspace, size_t workspace_bytes, void *stream);

/* learning.distances (scripts/learning.py:47-56): Euclidean distance, float64 by direct difference, of d_point[dim] to each of
 * d_rows[n_rows * dim] -> d_out[n_rows].  learning.closest_to (:59-66) is the row with the first smallest of them. */
int phm_distances(const double *d_point, const double *d_rows, int64_t n_rows, int dim, double *d_out, void *stream);

/* ---------------------------------------------------------------------------------------------
 * The whole hot path in one call (k = 4): count -> normalise -> score with the reference's default 'combo' method, i.e. what
 * scripts/phamer.py:131,139,194 do for one FASTA.  Same arguments as phm_kmer_count (d_seq, d_offsets) and phm_score (references,
 * centroids, outputs); d_counts (uint32[n_contigs * 256], required) receives the counts.  The histogram kernel emits the scorer's
 * query operands itself, so neither the feature matrix nor a preparation pass over the counts exists; results are bit-identical
 * to phm_kmer_count + phm_score_counts.  PHM_E_UNSUPPORTED outside the tensor-core shape (k_neighbors in {1, 3, 5}, both
 * centroid sets non-empty).
 * ------------------------------------------------------------------------------------------- */
size_t phm_count_score_workspace_bytes(int64_t n_contigs, int64_t n_bases, int64_t n_refs, int64_t n_cent_pos, int64_t n_cent_neg);
int phm_count_score(const uint8_t *d_seq, const int64_t *d_offsets, int64_t n_contigs,
                    const double *d_refs, int64_t n_refs, int64_t n_positive,
                    const double *d_cent_pos, int64_t n_cent_pos, const double *d_cent_neg, int64_t n_cent_neg,
                    int k_neighbors, uint32_t *d_counts, double *d_knn, double *d_kmeans, double *d_combo,
                    void *d_workspace, size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------------
 * FASTA ingest on the device (the caller / data-format row either side of the path, SURVEY.md 8(f) rank 3).  Replaces the
 * tokenisation kmer.count_file gets from Bio.SeqIO over a text-mode handle (scripts/kmer.py:131-139; scripts/fileIO.py:28-42):
 * a line ends at '\n', '\r' or "\r\n"; a record starts at a line beginning with '>', its sequence is every following line with
 * '\n', '\r' and ' ' removed (k-mers span line breaks, never records), text before the first '>' is ignored.  Two calls, so that
 * the caller can size the outputs in between:
 *
 *   phm_fasta_index    d_raw uint8[n_bytes] (16-byte aligned, allocation readable up to the next multiple of 16; what the bytes
 *                      past n_bytes hold does not matter)
 *                      -> d_result int64[4]: [0] records, [1] sequence bytes, [2] 1 if the file holds a control byte other than
 *                         '\n' '\r' (tab / VT / FF / 0x1C-0x1F among them; the reference strips those at line ends only: take
 *                         the host path for such files), [3] internal
 *   phm_fasta_extract  -> d_seq uint8[result[1]] sequence bytes end to end (ready for phm_kmer_count), d_offsets int64[records + 1],
 *                         d_header_pos int64[records] byte position of each record's '>' in the file (the host reads the titles
 *                         there); records beyond max_records are dropped: then d_offsets[max_records] is the start of the first
 *                         dropped record (the end of the last kept one), and nothing past d_offsets[max_records] or
 *                         d_header_pos[max_records - 1] is written
 * Both use the same d_workspace (phm_fasta_workspace_bytes), which must stay untouched between them.
 * ------------------------------------------------------------------------------------------- */
size_t phm_fasta_workspace_bytes(int64_t n_bytes);
int phm_fasta_index(const uint8_t *d_raw, int64_t n_bytes, int64_t *d_result, void *d_workspace, size_t workspace_bytes, void *stream);
int phm_fasta_extract(const uint8_t *d_raw, int64_t n_bytes, const int64_t *d_result, uint8_t *d_seq, int64_t *d_offsets,
                      int64_t *d_header_pos, int64_t max_records, const void *d_workspace, size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Lloyd iterations of k-means on the device (SURVEY.md 8(f) rank 4).  Replaces the iterations inside the reference's
 * KMeans(n_clusters = k, random_state = 10).fit(data).labels_ (learning.kmeans, scripts/learning.py:131-146; run twice per
 * scoring call, scripts/phamer.py:245-248).  The caller centres the data and seeds the centres exactly as scikit-learn does
 * (its own k-means++ routine), then:  E step = first argmin of |c|^2 - 2 x.c, M step = cluster means, stop when the labels
 * stop changing, when the summed squared centre shift is <= tol, or after max_iter; a final E step if the labels had not settled.
 *     d_x float64[n, dim] (dim <= 1024), d_centres float64[k, dim] in / out, d_labels int32[n] out
 *     h_info int64[3] (HOST) out: iterations, 1 if the labels settled, 1 if a cluster became empty (scikit-learn relocates empty
 *     clusters, this call does not: the caller must fall back to the host fit for that case)
 * SYNCHRONISES the stream once per iteration (convergence is decided on the host from 32 bytes).
 * ------------------------------------------------------------------------------------------- */
size_t phm_kmeans_workspace_bytes(int64_t n, int dim, int k);
int phm_kmeans_lloyd(const double *d_x, int64_t n, int dim, double *d_centres, int k, int max_iter, double tol,
                     int32_t *d_labels, int64_t *h_info, void *d_workspace, size_t workspace_bytes, void *stream);

/* Diagnostics of the last tensor-core phm_score call that used d_workspace (synchronises `stream`): rows that were
 * re-scored by the exhaustive float64 kernel because their candidate buffer overflowed; stats[0] = largest fraction of a
 * proven error interval used by a true ranking value (<= 1 means the proof held; only collected while option
 * "score_stats" is 1), stats[1] = largest |ranking value - exact| in squared-distance units (same condition), stats[2] =
 * rows whose neighbour vote needed exact re-measurement, stats[3] = rows whose candidate buffer overflowed and that were
 * settled by the second (listing) tensor-core pass.  The caller passes room for four floats. */
int phm_score_stats(const void *d_workspace, uint64_t *fallback_rows, float *max_rank_error, void *stream);

/* Tuning / path selection for experiments and tests (defaults are the measured best; every variant gives the same results).
 * Options: "hist_stride_k4" (2 | 1: 5-mer windows at every second base | plain 4-mers), "hist_stride_k5" (0 = automatic | 1 | 2: 6-mer windows in 16-bit packed counters),
 * "hist_warps_k5" (18 | 8: warps per CTA of the packed k = 5 table), "hist_warps_k6" (13 | 4), "hist_canonical_swizzle" (1 | 0: bank-swizzled table for the canonical fold at k = 5, 6),
 * "hist_tma" (0 | 1: sequence staged in shared memory by cp.async.bulk), "hist_plan" (1 | 0: records of 131 072 bases and more
 * are cut into tiles counted by different warps | every record is one work item),
 * "score_force_fallback" (1 = the first tensor-core pass keeps no candidate, so that every row takes the overflow road -- listing pass
 * or exhaustive kernels; this is how the tests exercise those kernels),
 * "score_list_pass" (0 = overflowed rows skip the listing pass and go to the exhaustive kernels),
 * "score_path" (0 = tensor cores when the shape allows, 1 = exhaustive float64 only, 2 = tensor cores or error),
 * "score_stats" (1 = collect error-interval diagnostics, slower), "time_kernels" (1 = bracket the hot kernels with CUDA
 * events for phm_last_kernel_ms). */
int phm_set_option(const char *name, int64_t value);

/* Kernels this library has launched in the calling process so far (bench.py reports the difference over its timed region). */
uint64_t phm_kernel_launches(void);

/* Mean device time (ms) of the launches (at most 64) of a hot kernel ("kmer_hist_kernel", "score_tc_kernel", "score_decide_kernel") since the previous
 * call for that kernel; needs option "time_kernels" = 1 before the launches.  Synchronises on the last of them. */
int phm_last_kernel_ms(const char *kernel, float *ms);

/* ---------------------------------------------------------------------------------------------
 * Synthetic workload (bench / tests only): contigs with lengths clip(round(exp(N(ln 10000, 1))), 1000,
 * 100000) (SURVEY.md 8(d) config 2), bases i.i.d. over ATGC with a per-contig GC fraction in
 * U(0.25, 0.75), counter-based RNG keyed by (seed, global contig index) so that a shard generated on
 * any rank equals the same rows of the single-GPU workload.
 *   phm_synth_lengths: d_lengths int64[n]   for contigs first_contig .. first_contig + n - 1
 *   phm_synth_bases:   fills d_seq[d_offsets[i] .. d_offsets[i+1])
 * ------------------------------------------------------------------------------------------- */
int phm_synth_lengths(uint64_t seed, int64_t first_contig, int64_t n_contigs, int64_t *d_lengths, void *stream);
int phm_synth_bases(uint64_t seed, int64_t first_contig, int64_t n_contigs, const int64_t *d_offsets,
                    uint8_t *d_seq, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* PHAMERS_B200_H */

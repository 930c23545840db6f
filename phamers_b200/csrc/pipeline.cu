// The whole hot path in one call: count -> (fused) normalise -> score.
//
// Replaces, for one batch of contigs, kmer.count_file's counting loop (reference scripts/kmer.py:137-139), kmer.normalize_counts
// (scripts/kmer.py:209-221, called at scripts/phamer.py:139) and phamer_scorer.score_points (scripts/phamer.py:177-195) with the
// default 'combo' method.  The reference features are prepared first (they fix the error-bound constants), then the histogram
// kernel writes, next to the counts, the tensor-core scorer's query operands of every contig from the table it still holds in
// shared memory, so the scoring stage starts directly with the contraction: no feature matrix and no preparation pass over
// the counts exist.  Results are bit-identical to phm_kmer_count followed by phm_score_counts (tests/test_gpu_score.py).
#include "score_common.cuh"

namespace phm {
int launch_count_emit(const uint8_t *seq, const int64_t *off, int64_t n, uint32_t *counts, void *ws, size_t ws_bytes,
                      tc::QueryEmit emit, cudaStream_t st);
}

using namespace phm;

static inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// layout: the scorer's workspace first (its size follows from the shapes), then the counting workspace, which takes whatever is left --
// its list of long work items is sized by the number of BASES, which this entry point is not told (see phm_kmer_count_workspace_bytes)
extern "C" size_t phm_count_score_workspace_bytes(int64_t n_contigs, int64_t n_bases, int64_t n_refs, int64_t n_cent_pos,
                                                  int64_t n_cent_neg) {
    return align256(phm_score_workspace_bytes(n_contigs, n_refs, n_cent_pos, n_cent_neg, 256)) +
           phm_kmer_count_workspace_bytes(n_contigs, n_bases, 4, 0);
}

extern "C" int phm_count_score(const uint8_t *d_seq, const int64_t *d_offsets, int64_t n_contigs,
                               const double *d_refs, int64_t n_refs, int64_t n_positive,
                               const double *d_cent_pos, int64_t n_cent_pos, const double *d_cent_neg, int64_t n_cent_neg,
                               int k_neighbors, uint32_t *d_counts, double *d_knn, double *d_kmeans, double *d_combo,
                               void *d_workspace, size_t workspace_bytes, void *stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    PHM_REQUIRE(n_contigs >= 0, "n_contigs must be >= 0");
    if (n_contigs == 0) return PHM_OK;
    PHM_REQUIRE(d_seq && d_offsets && d_counts && d_refs && d_workspace, "null pointer");
    PHM_REQUIRE(n_refs >= 1 && n_positive >= 0 && n_positive <= n_refs, "bad reference shape");
    PHM_REQUIRE((n_cent_pos == 0 || d_cent_pos) && (n_cent_neg == 0 || d_cent_neg), "null centroid pointer");
    if (!tc::score_tc_supported(256, k_neighbors, n_refs, n_cent_pos, n_cent_neg)) {
        set_error("phm_count_score needs the tensor-core shape: k_neighbors in {1, 3, 5} <= n_refs and both centroid sets");
        return PHM_E_UNSUPPORTED;
    }
    const size_t score_ws_bytes = align256(phm_score_workspace_bytes(n_contigs, n_refs, n_cent_pos, n_cent_neg, 256));
    if (workspace_bytes < phm_count_score_workspace_bytes(n_contigs, 0, n_refs, n_cent_pos, n_cent_neg)) {
        set_error("workspace too small");
        return PHM_E_WORKSPACE;
    }
    unsigned char *score_ws = static_cast<unsigned char *>(d_workspace);
    void *ws = score_ws + score_ws_bytes;
    const size_t count_ws = workspace_bytes - score_ws_bytes;

    ScoreArgs a;
    a.points = nullptr; a.point_counts = d_counts; a.n_points = n_contigs; a.dim = 256;
    a.refs = d_refs; a.n_refs = n_refs; a.n_positive = n_positive;
    a.cent_pos = d_cent_pos; a.n_cent_pos = n_cent_pos;
    a.cent_neg = d_cent_neg; a.n_cent_neg = n_cent_neg;
    a.norm_points = a.norm_refs = a.norm_cpos = a.norm_cneg = nullptr;
    a.out.k = k_neighbors;
    a.out.knn = d_knn; a.out.kmeans = d_kmeans; a.out.combo = d_combo;

    tc::QueryEmit emit;
    int rc = tc::score_tc_begin(a, score_ws, score_ws_bytes, st, &emit);                          // references: rho, pmax, B operand
    if (rc != PHM_OK) return rc;
    rc = launch_count_emit(d_seq, d_offsets, n_contigs, d_counts, ws, count_ws, emit, st);        // stage 1 + query operands
    if (rc != PHM_OK) return rc;
    return tc::score_tc_finish(a, score_ws, score_ws_bytes, st, true);                            // contraction, decision, fallback
}

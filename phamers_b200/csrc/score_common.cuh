// Declarations shared by the two scoring paths (score_exact.cu, score_tc.cu).
#pragma once
#include <cuda_fp16.h>
#include <math.h>

#include "phm_common.cuh"

namespace phm {

// Where a scoring call reports the rows that decided each query (phm_neighbors of the header): the k nearest references as rows
// of d_refs with their direct-difference distances, and the nearest centroid of each class.  Every member may be null.
struct NeighborOut {
    int64_t *ref_index = nullptr; double *ref_distance = nullptr;       // [n, k]
    int64_t *cent_index = nullptr; double *cent_distance = nullptr;     // [n, 2]: nearest positive, nearest negative
    __host__ __device__ bool any() const { return ref_index || ref_distance || cent_index || cent_distance; }
};

// What a scoring call writes for each row: the three scores (each may be null) and the neighbour report.
struct ScoreOut {
    int k;                                    // k_neighbors: report slots per row
    double *knn, *kmeans, *combo;
    NeighborOut nb;                           // all null: scores only
};

// ---- the rules of a row's outputs, the same on every road that finishes rows ----
__device__ __forceinline__ double knn_vote(int n_pos, int k) {
    return (2 * n_pos > k) ? 1.0 : -1.0;                               // 2 * (predict - 0.5), scripts/learning.py:128
}
// e_pos, e_neg: distances (not squares) to the nearest centroid of each class
__device__ __forceinline__ double kmeans_score(double e_pos, double e_neg) {
    return tanh((e_neg - e_pos) / (e_pos + e_neg));                    // scripts/phamer.py:206-209
}
__device__ __forceinline__ void put_scores(const ScoreOut &o, int64_t row, double knn, double km) {
    if (o.knn) o.knn[row] = knn;
    if (o.kmeans) o.kmeans[row] = km;
    if (o.combo) o.combo[row] = knn + km;                              // scripts/phamer.py:313
}
// one reported (index, distance) pair: slot `at` of the reference report (row * k + j) or of the centroid report (row * 2 + class)
__device__ __forceinline__ void put_neighbor(int64_t *index, double *distance, int64_t at, int64_t i, double d) {
    if (index) index[at] = i;
    if (distance) distance[at] = d;
}
// a NaN row reports index -1 and distance NaN everywhere
__device__ __forceinline__ void put_nan_row(const ScoreOut &o, int64_t row) {
    for (int j = 0; j < o.k; ++j) put_neighbor(o.nb.ref_index, o.nb.ref_distance, row * o.k + j, -1, NAN);
    for (int c = 0; c < 2; ++c) put_neighbor(o.nb.cent_index, o.nb.cent_distance, row * 2 + c, -1, NAN);
}

// ---- the order of neighbours: distance, then the lower index ----
// Roads that see candidates in ascending index (the exhaustive kernels, score_exact_kernel) keep with this comparator exactly
// what a strict '<' on the distance keeps: a later candidate never wins a tie.
template <typename I>
__device__ __forceinline__ bool nearer(double d, I i, double e, I j) { return d < e || (d == e && i < j); }

// insertion of (v, i) into a list of k entries sorted by nearer() (empty entries: INFINITY); drops the last entry
template <typename I>
__device__ __forceinline__ void list_insert(double *d, I *idx, int k, double v, I i) {
    if (!nearer(v, i, d[k - 1], idx[k - 1])) return;
    int s = k - 1;
    for (; s > 0 && nearer(v, i, d[s - 1], idx[s - 1]); --s) { d[s] = d[s - 1]; idx[s] = idx[s - 1]; }
    d[s] = v;
    idx[s] = i;
}

struct ScoreArgs {
    const double *points; int64_t n_points; int dim;
    const uint32_t *point_counts;             // optional: raw count rows instead of `points` (features = row / row sum, formed on the fly)
    const double *refs; int64_t n_refs; int64_t n_positive;
    const double *cent_pos; int64_t n_cent_pos;
    const double *cent_neg; int64_t n_cent_neg;
    const double *norm_points, *norm_refs, *norm_cpos, *norm_cneg;    // squared row norms (float64)
    ScoreOut out;
};

int launch_score_exact(const ScoreArgs &a, cudaStream_t st);
int launch_row_norms(const double *x, int64_t n_rows, int dim, double *out, cudaStream_t st);

namespace tc {

// ---- preparation of a query row for the tensor-core scorer (shared by tc_prep_rows_kernel and the histogram kernel's fused
// ---- emission, so that both produce the same bits) ----
struct PrepConsts {            // device-resident, written by the reference pass, read by whoever prepares query rows
    float rho;                 // max_j (dB_j + eps_acc (P_j + dB_j)) / P_j
    float pmax;                // max_j P_j
};
struct QueryEmit {             // where a producer of 256-wide count rows writes the scorer's query operands
    __half *op;                // [n, 256] centred, 2^12-scaled FP16 rows
    float *crow;               // [n] error constant C_row (NaN for an empty contig)
    double *cnorm;             // [n] |x - 1/256|^2
    uint32_t *total;           // [n] row total of the counts (the decision kernel forms count / total without a reduction)
    const PrepConsts *consts;
};
constexpr int PREP_DIM = 256;               // width of the FP16 operands
constexpr int CANON_DIM = 136;              // canonical 4-mer features: written into the first 136 operand columns, the rest stays zero
constexpr int KMER5_DIM = 1024;             // plain 5-mer features: operands 1024 wide (score_tc.cu streams the query tile)
constexpr int CANON5_DIM = 512;             // canonical 5-mer features: operands 512 wide
constexpr double PREP_SCALE = 4096.0;
// feature widths the tensor-core scorer takes
__host__ __device__ constexpr bool tc_width(int dim) {
    return dim == PREP_DIM || dim == CANON_DIM || dim == KMER5_DIM || dim == CANON5_DIM;
}
// a W-wide float64 row spread over a warp: lane l holds features l, l + 32, ... (NCH<W> chunks); in_row is false for the chunk
// slots beyond W, which read nothing and contribute exactly zero
template <int W> constexpr int NCH = (W + 31) / 32;
template <int W>
__device__ __forceinline__ bool in_row(int lane, int i) { return W % 32 == 0 || lane + 32 * i < W; }

__device__ __forceinline__ float float_up(double x) {           // a float that is >= x (x >= 0)
    float f = (float)x;
    return ((double)f >= x) ? f : __uint_as_float(__float_as_uint(f) + 1u);
}
// one feature of a W-wide row: FP16 operand element and the four running sums |x|^2, |x - u|^2, |A~ - A|^2, |A|^2 (scaled units),
// u = 1/W
template <int W = PREP_DIM>
__device__ __forceinline__ __half prep_accumulate(double x, double &s, double &sc, double &sd, double &sh) {
    const double xc = x - 1.0 / (double)W;
    const double t = xc * PREP_SCALE;
    const __half h = __float2half_rn((float)t);
    const double hv = (double)__half2float(h);
    s = fma(x, x, s);
    sc = fma(xc, xc, sc);
    sd = fma(t - hv, t - hv, sd);
    sh = fma(hv, hv, sh);
    return h;
}
// Sums of four doubles over the warp with 16 shuffles instead of 40: a butterfly that TRANSPOSES while it reduces (after the first
// exchange a lane carries two of the four values, after the second one), then three plain steps.  Every value is still reduced by
// the tree xor 16, 8, 4, 2, 1, so the sums have the bits the plain butterfly gives.  The results are valid in LANE 0 only.
__device__ __forceinline__ void warp_sum4(double &a, double &b, double &c, double &d, int lane) {
    const bool up = (lane & 16) != 0;
    const double k0 = (up ? c : a) + __shfl_xor_sync(FULL, up ? a : c, 16);
    const double k1 = (up ? d : b) + __shfl_xor_sync(FULL, up ? b : d, 16);
    const bool up2 = (lane & 8) != 0;
    double k = (up2 ? k1 : k0) + __shfl_xor_sync(FULL, up2 ? k0 : k1, 8);
    k += __shfl_xor_sync(FULL, k, 4);
    k += __shfl_xor_sync(FULL, k, 2);
    k += __shfl_xor_sync(FULL, k, 1);
    a = k;                                          // lane 0 holds a, lane 8 b, lane 16 c, lane 24 d
    b = __shfl_sync(FULL, k, 8);
    c = __shfl_sync(FULL, k, 16);
    d = __shfl_sync(FULL, k, 24);
}
__device__ __forceinline__ void warp_sum3(double &a, double &b, double &c, int lane) {
    const bool up = (lane & 16) != 0;
    const double k0 = (up ? c : a) + __shfl_xor_sync(FULL, up ? a : c, 16);
    const double k1 = (up ? 0.0 : b) + __shfl_xor_sync(FULL, up ? b : 0.0, 16);
    const bool up2 = (lane & 8) != 0;
    double k = (up2 ? k1 : k0) + __shfl_xor_sync(FULL, up2 ? k0 : k1, 8);
    k += __shfl_xor_sync(FULL, k, 4);
    k += __shfl_xor_sync(FULL, k, 2);
    k += __shfl_xor_sync(FULL, k, 1);
    a = k;
    b = __shfl_sync(FULL, k, 8);
    c = __shfl_sync(FULL, k, 16);
}
// err_j <= dA P_j + nA dB_j + eps_acc nA |B_j| + (FP32 roundings of nbs_j, of nbs_j - acc_j and of the fma)
//       <= P_j (dA + nA rho + 2^-21 (pmax + nA))        then 1 % on top for the FP32 arithmetic on the bounds
__device__ __forceinline__ float query_crow(double sc, double sd, double sh, float rho, float pmax) {
    const double dA = sqrt(sd) * (1.0 + 1e-12);
    const double nA = sqrt(sh) * (1.0 + 1e-12);
    const double c = (dA + nA * (double)rho + (double)(pmax + float_up(nA)) / 2097152.0) * 1.01;
    return isnan(sc) ? NAN : float_up(c);
}

int score_tc_begin(const ScoreArgs &a, void *ws, size_t ws_bytes, cudaStream_t st, QueryEmit *emit);
int score_tc_finish(const ScoreArgs &a, void *ws, size_t ws_bytes, cudaStream_t st, bool queries_prepared);
bool score_tc_supported(int dim, int k_neighbors, int64_t n_refs, int64_t n_cent_pos, int64_t n_cent_neg);
size_t score_tc_workspace_bytes(int64_t n_points, int64_t n_refs, int64_t n_cent_pos, int64_t n_cent_neg, int dim);
int score_tc(const ScoreArgs &a, void *ws, size_t ws_bytes, cudaStream_t st);
int score_tc_last_ms(float *ms);
int score_decide_last_ms(float *ms);
int score_tc_stats(const void *ws, unsigned long long *fallback_rows, float *max_rank_error, cudaStream_t st);
}  // namespace tc

extern int score_collect_stats;
extern int score_path;        // 0 = auto (tensor cores when supported), 1 = exact float64 only, 2 = tensor cores required

}  // namespace phm

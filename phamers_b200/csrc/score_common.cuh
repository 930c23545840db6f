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

struct ScoreArgs {
    const double *points; int64_t n_points; int dim;
    const uint32_t *point_counts;             // optional: raw count rows instead of `points` (features = row / row sum, formed on the fly)
    const double *refs; int64_t n_refs; int64_t n_positive;
    const double *cent_pos; int64_t n_cent_pos;
    const double *cent_neg; int64_t n_cent_neg;
    const double *norm_points, *norm_refs, *norm_cpos, *norm_cneg;    // squared row norms (float64)
    const int64_t *row_list;                  // optional: score only these rows
    const unsigned long long *n_rows_dev;     // optional: number of rows in row_list, read on the device
    int64_t n_rows;                           // rows to score (upper bound when n_rows_dev is set)
    int k_neighbors;
    double *knn, *kmeans, *combo;
    NeighborOut nb;                           // neighbour report (all null: scores only)
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
struct QueryEmit {             // where a producer of count rows writes the scorer's query operands
    __half *op;                // [n, 256] centred, 2^12-scaled FP16 rows
    float *crow;               // [n] error constant C_row (NaN for an empty contig)
    double *cnorm;             // [n] |x - 1/256|^2
    uint32_t *total;           // [n] row total of the counts (the decision kernel forms count / total without a reduction)
    const PrepConsts *consts;
};
constexpr int PREP_DIM = 256;
constexpr double PREP_SCALE = 4096.0;

__device__ __forceinline__ float float_up(double x) {           // a float that is >= x (x >= 0)
    float f = (float)x;
    return ((double)f >= x) ? f : __uint_as_float(__float_as_uint(f) + 1u);
}
// one feature: FP16 operand element and the four running sums |x|^2, |x - u|^2, |A~ - A|^2, |A|^2 (scaled units)
__device__ __forceinline__ __half prep_accumulate(double x, double &s, double &sc, double &sd, double &sh) {
    const double xc = x - 1.0 / (double)PREP_DIM;
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
size_t score_tc_workspace_bytes(int64_t n_points, int64_t n_refs, int64_t n_cent_pos, int64_t n_cent_neg);
int score_tc(const ScoreArgs &a, void *ws, size_t ws_bytes, cudaStream_t st, int *kernels_launched);
int score_tc_last_ms(float *ms);
int score_decide_last_ms(float *ms);
int score_tc_stats(const void *ws, unsigned long long *fallback_rows, float *max_rank_error, cudaStream_t st);
}  // namespace tc

extern int score_collect_stats;
extern int score_path;        // 0 = auto (tensor cores when supported), 1 = exact float64 only, 2 = tensor cores required

}  // namespace phm

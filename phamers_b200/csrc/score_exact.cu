// K4/K5 exact path: float64 brute-force scorer.
//
// Replaces learning.knn (reference scripts/learning.py:118-128 -> scikit-learn brute-force kNN, which itself ranks by
// the float64 expansion |x|^2 - 2 x.y + |y|^2), learning.closest_to (:59-66) and phamer_scorer.proximity_metric
// (scripts/phamer.py:198-210).  Every (query, reference) and (query, centroid) squared distance is formed in float64
// from a register-tiled x.y; the k nearest references vote, the two best centroids of each class are re-measured by
// direct difference (as np.linalg.norm(point - centroid) does) and the nearer one enters tanh((e_n - e_p)/(e_p + e_n)).
//
// This kernel is the always-correct path: the tensor-core scorer (score_tc.cu) uses it for the rows whose candidate
// buffer overflows, and the tests use it to cross-check the tensor-core path at sizes the CPU oracle cannot reach.
#include <math.h>

#include "score_common.cuh"

namespace phm {

constexpr int TQ = 64;        // queries per CTA
constexpr int TR = 64;        // reference columns per tile
constexpr int DK = 16;        // feature chunk
constexpr int KNN_MAX = 15;

__global__ void row_norms_kernel(const double *__restrict__ x, int64_t n_rows, int dim, double *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < n_rows; r += n_warps) {
        double s = 0.0;
        for (int d = lane; d < dim; d += 32) {
            const double v = x[r * dim + d];
            s = fma(v, v, s);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(FULL, s, o);
        if (lane == 0) out[r] = s;
    }
}

struct ExactSmem {
    double As[DK][TQ + 4];
    double Bs[DK][TR + 4];
    double Ds[TQ][TR + 1];
    double col_norm[TR];
    double knn_d[TQ][KNN_MAX + 1];
    double cen_d[TQ][4];      // [0..1] two best positive centroids, [2..3] two best negative
    int64_t qrow[TQ];
    int knn_i[TQ][KNN_MAX + 1];
    int cen_i[TQ][4];
};

__device__ __forceinline__ const double *column_row(const ScoreArgs &a, int64_t col, double *norm) {
    if (col < a.n_refs) { *norm = a.norm_refs[col]; return a.refs + col * a.dim; }
    col -= a.n_refs;
    if (col < a.n_cent_pos) { *norm = a.norm_cpos[col]; return a.cent_pos + col * a.dim; }
    col -= a.n_cent_pos;
    *norm = a.norm_cneg[col];
    return a.cent_neg + col * a.dim;
}

__device__ __forceinline__ double direct_distance(const double *p, const double *c, int dim) {
    double s = 0.0;
    for (int d = 0; d < dim; ++d) {
        const double t = p[d] - c[d];
        s = fma(t, t, s);
    }
    return sqrt(s);
}

// Neighbour report of one row.  The selection ranks by the norm expansion; the k references it kept are re-measured by direct
// difference and ordered by (distance, index), and the nearer of the two re-measured centroids of each class is reported (lower
// index on ties).  At a near tie (a gap below the expansion's rounding) the selection may keep the other member of the tie than
// the tensor-core path does.  A NaN row reports index -1 and distance NaN everywhere.
__device__ void exact_neighbors(const ScoreArgs &a, int64_t q, bool nan_row, const int (&ki)[KNN_MAX + 1], const int (&ci)[4]) {
    const ScoreOut &o = a.out;
    if (nan_row) { put_nan_row(o, q); return; }
    const int kn = o.k;
    const double *p = a.points + q * a.dim;
    double d[KNN_MAX];
    int64_t id[KNN_MAX];
    for (int j = 0; j < kn; ++j) {
        const bool ok = ki[j] >= 0;
        id[j] = ok ? ki[j] : -1;
        d[j] = ok ? direct_distance(p, a.refs + (int64_t)ki[j] * a.dim, a.dim) : NAN;
        for (int s = j; s > 0 && nearer(d[s], id[s], d[s - 1], id[s - 1]); --s) {
            const double td = d[s]; d[s] = d[s - 1]; d[s - 1] = td;
            const int64_t ti = id[s]; id[s] = id[s - 1]; id[s - 1] = ti;
        }
    }
    for (int j = 0; j < kn; ++j) put_neighbor(o.nb.ref_index, o.nb.ref_distance, q * kn + j, id[j], d[j]);
    for (int c = 0; c < 2; ++c) {
        const double *cent = c ? a.cent_neg : a.cent_pos;
        int64_t best = -1;
        double bd = NAN;
        for (int j = 0; j < 2; ++j) {
            const int i = ci[2 * c + j];
            if (i < 0) continue;
            const double e = direct_distance(p, cent + (int64_t)i * a.dim, a.dim);
            if (best < 0 || nearer(e, (int64_t)i, bd, best)) { best = i; bd = e; }
        }
        put_neighbor(o.nb.cent_index, o.nb.cent_distance, q * 2 + c, best, bd);
    }
}

__global__ void __launch_bounds__(256) score_exact_kernel(ScoreArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    ExactSmem &sm = *reinterpret_cast<ExactSmem *>(smem_raw);
    auto &As = sm.As; auto &Bs = sm.Bs; auto &Ds = sm.Ds; auto &col_norm = sm.col_norm;
    auto &knn_d = sm.knn_d; auto &knn_i = sm.knn_i; auto &cen_d = sm.cen_d; auto &cen_i = sm.cen_i;
    auto &qrow = sm.qrow;

    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    const int64_t q0 = (int64_t)blockIdx.x * TQ;
    const int64_t n_cols = a.n_refs + a.n_cent_pos + a.n_cent_neg;
    const int kn = a.out.k;

    if (tid < TQ) {
        const int64_t r = q0 + tid;
        qrow[tid] = (r < a.n_points) ? r : -1;
        for (int j = 0; j <= KNN_MAX; ++j) { knn_d[tid][j] = INFINITY; knn_i[tid][j] = -1; }
        for (int j = 0; j < 4; ++j) { cen_d[tid][j] = INFINITY; cen_i[tid][j] = -1; }
    }
    __syncthreads();

    for (int64_t c0 = 0; c0 < n_cols; c0 += TR) {
        double acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;

        const int lrow = tid >> 2;           // 0..63: which query / column this thread stages
        const int lseg = (tid & 3) * 4;      // 4 consecutive features
        const int64_t my_q = qrow[lrow];
        const int64_t my_c = c0 + lrow;
        double cn = 0.0;
        const double *crow = (my_c < n_cols) ? column_row(a, my_c, &cn) : nullptr;
        if ((tid & 3) == 0) col_norm[lrow] = crow ? cn : INFINITY;

        for (int d0 = 0; d0 < a.dim; d0 += DK) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int d = d0 + lseg + i;
                As[lseg + i][lrow] = (my_q >= 0 && d < a.dim) ? a.points[my_q * a.dim + d] : 0.0;
                Bs[lseg + i][lrow] = (crow && d < a.dim) ? crow[d] : 0.0;
            }
            __syncthreads();
#pragma unroll
            for (int kk = 0; kk < DK; ++kk) {
                double av[4], bv[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) { av[i] = As[kk][ty * 4 + i]; bv[i] = Bs[kk][tx * 4 + i]; }
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = fma(av[i], bv[j], acc[i][j]);
            }
            __syncthreads();
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int64_t q = qrow[ty * 4 + i];
            const double qn = (q >= 0) ? a.norm_points[q] : 0.0;
#pragma unroll
            for (int j = 0; j < 4; ++j) Ds[ty * 4 + i][tx * 4 + j] = qn + col_norm[tx * 4 + j] - 2.0 * acc[i][j];
        }
        __syncthreads();

        if (tid < TQ && qrow[tid] >= 0) {
            for (int j = 0; j < TR; ++j) {
                const int64_t col = c0 + j;
                if (col >= n_cols) break;
                const double d = Ds[tid][j];
                if (col < a.n_refs) {
                    list_insert(knn_d[tid], knn_i[tid], kn, d, (int)col);
                } else {
                    const bool neg = col >= a.n_refs + a.n_cent_pos;
                    const int b = neg ? 2 : 0;
                    const int ci = (int)(col - a.n_refs - (neg ? a.n_cent_pos : 0));
                    if (d < cen_d[tid][b]) {
                        cen_d[tid][b + 1] = cen_d[tid][b]; cen_i[tid][b + 1] = cen_i[tid][b];
                        cen_d[tid][b] = d; cen_i[tid][b] = ci;
                    } else if (d < cen_d[tid][b + 1]) {
                        cen_d[tid][b + 1] = d; cen_i[tid][b + 1] = ci;
                    }
                }
            }
        }
        __syncthreads();
    }

    if (tid < TQ && qrow[tid] >= 0) {
        const int64_t q = qrow[tid];
        const double qn = a.norm_points[q];
        double knn = NAN, km = NAN;
        if (!isnan(qn)) {
            int pos = 0;
            for (int j = 0; j < kn; ++j) pos += (knn_i[tid][j] >= 0 && knn_i[tid][j] < a.n_positive);
            knn = knn_vote(pos, kn);
            if (a.n_cent_pos > 0 && a.n_cent_neg > 0) {
                const double *p = a.points + q * a.dim;
                double e_pos = INFINITY, e_neg = INFINITY;
                for (int j = 0; j < 2; ++j) {
                    if (cen_i[tid][j] >= 0) e_pos = fmin(e_pos, direct_distance(p, a.cent_pos + (int64_t)cen_i[tid][j] * a.dim, a.dim));
                    if (cen_i[tid][2 + j] >= 0) e_neg = fmin(e_neg, direct_distance(p, a.cent_neg + (int64_t)cen_i[tid][2 + j] * a.dim, a.dim));
                }
                km = kmeans_score(e_pos, e_neg);
            }
        }
        put_scores(a.out, q, knn, km);
        if (a.out.nb.any()) exact_neighbors(a, q, isnan(qn), knn_i[tid], cen_i[tid]);
    }
}

int launch_score_exact(const ScoreArgs &a, cudaStream_t st) {
    if (a.n_points == 0) return PHM_OK;
    const int64_t blocks = (a.n_points + TQ - 1) / TQ;
    PHM_CUDA_CHECK(cudaFuncSetAttribute(score_exact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ExactSmem)));
    score_exact_kernel<<<(unsigned)blocks, 256, sizeof(ExactSmem), st>>>(a);
    PHM_LAUNCH_CHECK();
    return PHM_OK;
}

int launch_row_norms(const double *x, int64_t n_rows, int dim, double *out, cudaStream_t st) {
    if (n_rows == 0) return PHM_OK;
    int64_t blocks = (n_rows + 7) / 8;
    if (blocks > 148 * 16) blocks = 148 * 16;
    row_norms_kernel<<<(unsigned)blocks, 256, 0, st>>>(x, n_rows, dim, out);
    PHM_LAUNCH_CHECK();
    return PHM_OK;
}

// learning.distances (scripts/learning.py:47-56): Euclidean distance of one point to every row, float64 by direct difference
// (the arithmetic every exact path of the scorer uses).  One warp per row.
__global__ void __launch_bounds__(256) distances_kernel(const double *__restrict__ point, const double *__restrict__ rows, int64_t n_rows,
                                                        int dim, double *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < n_rows; r += n_warps) {
        double acc = 0.0;
        for (int d = lane; d < dim; d += 32) {
            const double t = point[d] - rows[r * dim + d];
            acc = fma(t, t, acc);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(FULL, acc, o);
        if (lane == 0) out[r] = sqrt(acc);
    }
}

// kmer.normalize_counts for rows that are not exact 32-bit counts (summed genome counts, features): row / row sum in float64.
// The row sum is accumulated in float64 lane by lane and then across the warp; for integer-valued rows below 2^53 it is exact
// and the result equals numpy's, for other rows it can differ from numpy's pairwise sum in the last bit.
__global__ void __launch_bounds__(256) normalize_rows_kernel(const double *__restrict__ in, int64_t n_rows, int64_t bins, double *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < n_rows; r += n_warps) {
        double total = 0.0;
        for (int64_t b = lane; b < bins; b += 32) total += in[r * bins + b];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(FULL, total, o);
        for (int64_t b = lane; b < bins; b += 32) out[r * bins + b] = in[r * bins + b] / total;
    }
}

}  // namespace phm

namespace phm { int score_path = 0; }

using namespace phm;


extern "C" size_t phm_score_workspace_bytes(int64_t n_points, int64_t n_refs, int64_t n_cent_pos, int64_t n_cent_neg, int dim) {
    const size_t exact = (size_t)(n_points + n_refs + n_cent_pos + n_cent_neg + 8) * sizeof(double);
    if (tc::tc_width(dim)) {                    // 256 or 136: 256-wide FP16 operands; 512 or 1024: operands of that width
        const size_t tcb = tc::score_tc_workspace_bytes(n_points, n_refs, n_cent_pos, n_cent_neg, dim);
        return tcb > exact ? tcb : exact;
    }
    return exact;
}

static int score_any(const double *d_points, const uint32_t *d_point_counts, int64_t n_points, int dim,
                     const double *d_refs, int64_t n_refs, int64_t n_positive,
                     const double *d_cent_pos, int64_t n_cent_pos, const double *d_cent_neg, int64_t n_cent_neg,
                     int k_neighbors, double *d_knn, double *d_kmeans, double *d_combo, const phm_neighbors *nb,
                     void *d_workspace, size_t workspace_bytes, void *stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    PHM_REQUIRE(n_points >= 0 && dim > 0, "bad query shape");
    PHM_REQUIRE(n_refs >= 1 && n_positive >= 0 && n_positive <= n_refs, "bad reference shape");
    PHM_REQUIRE(k_neighbors >= 1 && k_neighbors <= KNN_MAX && k_neighbors <= n_refs, "k_neighbors must be 1..15 and <= n_refs");
    PHM_REQUIRE(n_cent_pos >= 0 && n_cent_neg >= 0, "bad centroid shape");
    if (n_points == 0) return PHM_OK;
    PHM_REQUIRE((d_points || d_point_counts) && d_refs, "null pointer");
    PHM_REQUIRE((n_cent_pos == 0 || d_cent_pos) && (n_cent_neg == 0 || d_cent_neg), "null centroid pointer");
    PHM_REQUIRE(d_workspace != nullptr, "d_workspace is null");
    if (workspace_bytes < phm_score_workspace_bytes(n_points, n_refs, n_cent_pos, n_cent_neg, dim)) {
        set_error("workspace too small");
        return PHM_E_WORKSPACE;
    }
    ScoreArgs a;
    a.points = d_points; a.point_counts = d_point_counts; a.n_points = n_points; a.dim = dim;
    a.refs = d_refs; a.n_refs = n_refs; a.n_positive = n_positive;
    a.cent_pos = d_cent_pos; a.n_cent_pos = n_cent_pos;
    a.cent_neg = d_cent_neg; a.n_cent_neg = n_cent_neg;
    a.out.k = k_neighbors;
    a.out.knn = d_knn; a.out.kmeans = d_kmeans; a.out.combo = d_combo;
    if (nb) {
        a.out.nb.ref_index = nb->d_ref_index; a.out.nb.ref_distance = nb->d_ref_distance;
        a.out.nb.cent_index = nb->d_centroid_index; a.out.nb.cent_distance = nb->d_centroid_distance;
    }

    const bool tc_ok = tc::score_tc_supported(dim, k_neighbors, n_refs, n_cent_pos, n_cent_neg);
    if (score_path == 2 && !tc_ok) {
        set_error("tensor-core scoring needs dim = 256, 136, 512 or 1024, k_neighbors in {1, 3, 5} and both centroid sets");
        return PHM_E_UNSUPPORTED;
    }
    // Float64 feature rows 136, 512 or 1024 wide keep the exhaustive kernel unless tensor cores are required: it was their road
    // before the tensor-core road took those widths, and the two roads order exact distance ties differently (norm expansion against
    // direct difference), so this keeps phm_score's answers at those widths as they were.  Count rows (phm_score_counts) take the
    // tensor cores.
    const bool tc_auto = tc_ok && (dim == tc::PREP_DIM || d_point_counts != nullptr);
    if ((score_path == 0 && tc_auto) || (score_path == 2 && tc_ok)) return tc::score_tc(a, d_workspace, workspace_bytes, st);
    if (d_point_counts) {
        set_error("scoring from raw counts needs the tensor-core path (dim = 256, 136, 512 or 1024, k_neighbors in {1, 3, 5}, both centroid "
                  "sets); normalise first (phm_normalize_counts) and call phm_score");
        return PHM_E_UNSUPPORTED;
    }

    double *ws = static_cast<double *>(d_workspace);
    double *np_ = ws, *nr = np_ + n_points, *ncp = nr + n_refs, *ncn = ncp + n_cent_pos;
    a.norm_points = np_; a.norm_refs = nr; a.norm_cpos = ncp; a.norm_cneg = ncn;
    int rc;
    if ((rc = launch_row_norms(d_points, n_points, dim, np_, st)) != PHM_OK) return rc;
    if ((rc = launch_row_norms(d_refs, n_refs, dim, nr, st)) != PHM_OK) return rc;
    if ((rc = launch_row_norms(d_cent_pos, n_cent_pos, dim, ncp, st)) != PHM_OK) return rc;
    if ((rc = launch_row_norms(d_cent_neg, n_cent_neg, dim, ncn, st)) != PHM_OK) return rc;
    return launch_score_exact(a, st);
}

extern "C" int phm_score(const double *d_points, int64_t n_points, int dim,
                         const double *d_refs, int64_t n_refs, int64_t n_positive,
                         const double *d_cent_pos, int64_t n_cent_pos, const double *d_cent_neg, int64_t n_cent_neg,
                         int k_neighbors, double *d_knn, double *d_kmeans, double *d_combo,
                         void *d_workspace, size_t workspace_bytes, void *stream) {
    PHM_REQUIRE(d_points != nullptr || n_points == 0, "d_points is null");
    return score_any(d_points, nullptr, n_points, dim, d_refs, n_refs, n_positive, d_cent_pos, n_cent_pos, d_cent_neg, n_cent_neg,
                     k_neighbors, d_knn, d_kmeans, d_combo, nullptr, d_workspace, workspace_bytes, stream);
}

// Stages 2 + 3 fused: the query features are never materialised, every kernel forms count / row total on the fly.
extern "C" int phm_score_counts(const uint32_t *d_counts, int64_t n_points, int dim,
                                const double *d_refs, int64_t n_refs, int64_t n_positive,
                                const double *d_cent_pos, int64_t n_cent_pos, const double *d_cent_neg, int64_t n_cent_neg,
                                int k_neighbors, double *d_knn, double *d_kmeans, double *d_combo,
                                void *d_workspace, size_t workspace_bytes, void *stream) {
    PHM_REQUIRE(d_counts != nullptr || n_points == 0, "d_counts is null");
    return score_any(nullptr, d_counts, n_points, dim, d_refs, n_refs, n_positive, d_cent_pos, n_cent_pos, d_cent_neg, n_cent_neg,
                     k_neighbors, d_knn, d_kmeans, d_combo, nullptr, d_workspace, workspace_bytes, stream);
}

extern "C" int phm_score_neighbors(const double *d_points, int64_t n_points, int dim,
                                   const double *d_refs, int64_t n_refs, int64_t n_positive,
                                   const double *d_cent_pos, int64_t n_cent_pos, const double *d_cent_neg, int64_t n_cent_neg,
                                   int k_neighbors, double *d_knn, double *d_kmeans, double *d_combo, const phm_neighbors *nb,
                                   void *d_workspace, size_t workspace_bytes, void *stream) {
    PHM_REQUIRE(d_points != nullptr || n_points == 0, "d_points is null");
    return score_any(d_points, nullptr, n_points, dim, d_refs, n_refs, n_positive, d_cent_pos, n_cent_pos, d_cent_neg, n_cent_neg,
                     k_neighbors, d_knn, d_kmeans, d_combo, nb, d_workspace, workspace_bytes, stream);
}

extern "C" int phm_score_counts_neighbors(const uint32_t *d_counts, int64_t n_points, int dim,
                                          const double *d_refs, int64_t n_refs, int64_t n_positive,
                                          const double *d_cent_pos, int64_t n_cent_pos, const double *d_cent_neg, int64_t n_cent_neg,
                                          int k_neighbors, double *d_knn, double *d_kmeans, double *d_combo, const phm_neighbors *nb,
                                          void *d_workspace, size_t workspace_bytes, void *stream) {
    PHM_REQUIRE(d_counts != nullptr || n_points == 0, "d_counts is null");
    return score_any(nullptr, d_counts, n_points, dim, d_refs, n_refs, n_positive, d_cent_pos, n_cent_pos, d_cent_neg, n_cent_neg,
                     k_neighbors, d_knn, d_kmeans, d_combo, nb, d_workspace, workspace_bytes, stream);
}

// Diagnostics of the last tensor-core phm_score call that used this workspace (synchronises the stream).
extern "C" int phm_score_stats(const void *d_workspace, uint64_t *fallback_rows, float *max_rank_error, void *stream) {
    PHM_REQUIRE(d_workspace && fallback_rows && max_rank_error, "null pointer");
    unsigned long long fb = 0;                  // max_rank_error points at 3 floats: absolute, relative, rows re-measured
    int rc = tc::score_tc_stats(d_workspace, &fb, max_rank_error, static_cast<cudaStream_t>(stream));
    *fallback_rows = fb;
    return rc;
}

extern "C" int phm_distances(const double *d_point, const double *d_rows, int64_t n_rows, int dim, double *d_out, void *stream) {
    PHM_REQUIRE(n_rows >= 0 && dim > 0, "bad shape");
    if (n_rows == 0) return PHM_OK;
    PHM_REQUIRE(d_point != nullptr && d_rows != nullptr && d_out != nullptr, "null pointer");
    int64_t blocks = (n_rows + 7) / 8;
    if (blocks > (int64_t)sm_count() * 16) blocks = (int64_t)sm_count() * 16;
    distances_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(d_point, d_rows, n_rows, dim, d_out);
    PHM_LAUNCH_CHECK();
    return PHM_OK;
}

extern "C" int phm_normalize_rows(const double *d_rows, int64_t n_rows, int64_t bins, double *d_out, void *stream) {
    PHM_REQUIRE(n_rows >= 0 && bins > 0, "bad shape");
    if (n_rows == 0) return PHM_OK;
    PHM_REQUIRE(d_rows != nullptr && d_out != nullptr, "null pointer");
    int64_t blocks = (n_rows + 7) / 8;
    if (blocks > (int64_t)sm_count() * 16) blocks = (int64_t)sm_count() * 16;
    normalize_rows_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(d_rows, n_rows, bins, d_out);
    PHM_LAUNCH_CHECK();
    return PHM_OK;
}

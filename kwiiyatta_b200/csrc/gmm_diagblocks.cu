// Joint-GMM EM with diagonal covariance blocks (covariance_type 'diagonal_blocks'), FP64 on the
// CUDA cores, for sm_100a.
//
// The joint vector is z = [x, y] with D = 2 Dh, and each of the four Dh x Dh blocks Sxx, Sxy, Syx,
// Syy of a component's covariance is diagonal.  The only coupling left is between x_d and y_d, so
// the model is Dh independent 2 x 2 Gaussians per component and every step works per feature pair
// (restated in oracle/gmm_diagblocks_ref.py; layouts in include/kwiiyatta_b200.h):
//
//   E-step   u = x_d - mu_d, v = y_d - mu_{Dh+d};  [u v] U_kd = [a u, b u + c v]
//            wlp[n,k] = -1/2 (D log 2pi + sum_d (a u)^2 + (b u + c v)^2) + log|U_k| + log w_k
//            resp = exp(wlp - logsumexp_k wlp);  sum_n logsumexp -> lower bound
//   M-step   n_k, sum r (z - c_k), per pair sum r u^2, sum r u v, sum r v^2 around the centres c_k,
//            partials reduced in a fixed order (bitwise reproducible)
//   finalize weights, means, per pair covariance (+reg I), 2 x 2 Cholesky and its inverse factor
//            U = [[a, b], [0, c]] (Sigma^-1 = U U^T, sklearn's upper precision Cholesky), log|U|.
#include <cfloat>

#include "common.cuh"

namespace kw {

constexpr int DB_FT = 64;         // frames per CTA tile in the E-step
constexpr int DB_THREADS = 256;
constexpr int DB_FIN_THREADS = 128;   // >= GMM_MAX_DIM / 2 feature pairs
static_assert(DB_FIN_THREADS >= GMM_MAX_DIM / 2, "one finaliser thread per feature pair");

__host__ __device__ static inline size_t db_stats_block(int D) {
    return 1 + (size_t)D + 3 * (size_t)(D / 2);
}

// ---------------------------------------------------------------------------------------
// E-step.  CTA = 64 frames x all K components.  The frame tile sits in shared memory; thread
// (f = tid % 64, g = tid / 64) evaluates frame f against components g, g + 4, ..., so a warp reads
// one component's means and factors at a time (broadcast loads).  The weighted log-probabilities
// go to resp, and the CTA normalises its own frames from there: one thread per frame, as in
// gmm_estep_kernel.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(DB_THREADS)
gmm_db_estep_kernel(long long N, long long Npad, const double* __restrict__ X, int K, int D,
                    const double* __restrict__ means, const double* __restrict__ factors,
                    const double* __restrict__ aux, double* __restrict__ resp,
                    double* __restrict__ lse_partial, double* __restrict__ lse_frame) {
    extern __shared__ double xs[];   // DB_FT x (D + 1)
    __shared__ double frame_lse[DB_FT];
    const int Dh = D / 2, XS = D + 1;
    const int tid = threadIdx.x;
    const long long n0 = (long long)blockIdx.x * DB_FT;
    const double LOG2PI = 1.8378770664093453;

    for (int e = tid; e < DB_FT * D; e += DB_THREADS) {
        const int f = e / D, dd = e - f * D;
        const long long n = n0 + f;
        xs[f * XS + dd] = (n < N) ? X[n * D + dd] : 0.0;
    }
    __syncthreads();
    {
        const int f = tid & (DB_FT - 1);
        const long long n = n0 + f;
        const double* x = xs + f * XS;
        for (int k = tid / DB_FT; k < K; k += DB_THREADS / DB_FT) {
            const double* mu = means + (size_t)k * D;
            const double* U = factors + (size_t)k * 3 * Dh;
            double q = 0.0;
#pragma unroll 4
            for (int d = 0; d < Dh; ++d) {
                const double u = x[d] - mu[d], v = x[Dh + d] - mu[Dh + d];
                const double y0 = U[3 * d] * u;
                const double y1 = fma(U[3 * d + 1], u, U[3 * d + 2] * v);
                q = fma(y0, y0, q);
                q = fma(y1, y1, q);
            }
            const double wlp = (-0.5 * ((double)D * LOG2PI + q) + aux[2 * k]) + aux[2 * k + 1];
            if (n < N) __stcg(resp + (size_t)k * Npad + n, wlp);
        }
    }
    __syncthreads();
    if (tid < DB_FT) {
        const long long n = n0 + tid;
        double lse = 0.0;
        if (n < N) {
            double* col = resp + n;
            double mx = -CUDART_INF;
            for (int k = 0; k < K; ++k) mx = fmax(mx, __ldcg(col + (size_t)k * Npad));
            double sum = 0.0;
            for (int k = 0; k < K; ++k) sum += exp(__ldcg(col + (size_t)k * Npad) - mx);
            lse = log(sum) + mx;
            for (int k = 0; k < K; ++k)
                col[(size_t)k * Npad] = exp(__ldcg(col + (size_t)k * Npad) - lse);
            if (lse_frame != nullptr) lse_frame[n] = lse;
        }
        frame_lse[tid] = lse;
    }
    __syncthreads();
    if (tid == 0) {
        double t = 0.0;
        for (int f = 0; f < DB_FT; ++f) t += frame_lse[f];
        lse_partial[blockIdx.x] = t;
    }
}

// ---------------------------------------------------------------------------------------
// M-step statistics: grid (K, chunks).  Thread (p = tid % Dh, g = tid / Dh) owns feature pair p
// for the frames g, g + G, ... of the chunk (G = 256 / Dh groups), skipping r <= resp_floor; the
// groups are then summed in group order.  partial layout: [chunk][k][db_stats_block(D)].
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(DB_THREADS)
gmm_db_mstats_kernel(long long N, long long Npad, const double* __restrict__ X, int K, int D,
                     const double* __restrict__ respT, const double* __restrict__ centres,
                     double* __restrict__ partial, long long frames_per_chunk, double resp_floor) {
    __shared__ double red[5][DB_THREADS];
    __shared__ double nred[DB_THREADS];
    const int Dh = D / 2, G = DB_THREADS / Dh;
    const int tid = threadIdx.x;
    const int p = tid % Dh, g = tid / Dh;
    const int k = blockIdx.x;
    const long long n_begin = (long long)blockIdx.y * frames_per_chunk;
    const long long n_end = min(N, n_begin + frames_per_chunk);
    const double* rk = respT + (size_t)k * Npad;
    double su = 0.0, sv = 0.0, suu = 0.0, suv = 0.0, svv = 0.0, sn = 0.0;
    if (g < G) {
        const double cu = centres[(size_t)k * D + p], cv = centres[(size_t)k * D + Dh + p];
#pragma unroll 4
        for (long long n = n_begin + g; n < n_end; n += G) {
            const double r = rk[n];
            if (r > resp_floor) {
                const double u = X[n * D + p] - cu, v = X[n * D + Dh + p] - cv;
                const double ru = r * u, rv = r * v;
                su += ru;
                sv += rv;
                suu = fma(ru, u, suu);
                suv = fma(ru, v, suv);
                svv = fma(rv, v, svv);
                sn += r;
            }
        }
    }
    red[0][tid] = su;
    red[1][tid] = sv;
    red[2][tid] = suu;
    red[3][tid] = suv;
    red[4][tid] = svv;
    nred[tid] = sn;
    __syncthreads();
    double* out = partial + ((size_t)blockIdx.y * K + k) * db_stats_block(D);
    if (tid < Dh) {
        double t[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
        for (int h = 0; h < G; ++h)
#pragma unroll
            for (int s = 0; s < 5; ++s) t[s] += red[s][h * Dh + tid];
        out[1 + tid] = t[0];
        out[1 + Dh + tid] = t[1];
        double* so = out + 1 + D + 3 * tid;
        so[0] = t[2];
        so[1] = t[3];
        so[2] = t[4];
    }
    if (tid == 0) {
        double t = 0.0;
        for (int h = 0; h < G; ++h) t += nred[h * Dh];   // pair 0 of each group carries n_k
        out[0] = t;
    }
}

// stats[e] = sum over chunks (fixed order) of the partials.
__global__ void gmm_db_reduce_partials_kernel(size_t total, int chunks,
                                              const double* __restrict__ partial,
                                              double* __restrict__ stats) {
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total;
         e += (size_t)gridDim.x * blockDim.x) {
        double s = 0.0;
        for (int c = 0; c < chunks; ++c) s += partial[(size_t)c * total + e];
        stats[e] = s;
    }
}

// ---------------------------------------------------------------------------------------
// Finalize: one CTA per component, one thread per feature pair.  from_stats = 1: parameters
// from sufficient statistics (as gmm_finalize_kernel); from_stats = 0: the factors and aux of
// given covariances and weights.  info[k] = 0, or the 1-based index (in the expanded D x D matrix)
// of the first non-positive Cholesky pivot.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(DB_FIN_THREADS)
gmm_db_finalize_kernel(int K, int D, double reg_covar, int weight_norm, int from_stats,
                       const double* __restrict__ stats, const double* __restrict__ centres,
                       double* __restrict__ weights, double* __restrict__ means,
                       double* __restrict__ cov, double* __restrict__ factors,
                       double* __restrict__ aux, int32_t* __restrict__ info) {
    __shared__ double sh_ld[DB_FIN_THREADS];
    __shared__ int sh_bad[DB_FIN_THREADS];
    const int Dh = D / 2;
    const int k = blockIdx.x, p = threadIdx.x;
    double* ck = cov + (size_t)k * 3 * Dh;
    double wk;
    if (from_stats) {
        const size_t sb = db_stats_block(D);
        const double* st = stats + (size_t)k * sb;
        const double EPS10 = 10.0 * DBL_EPSILON;
        const double nk = st[0] + EPS10;
        double denom;
        if (weight_norm == 1) {
            denom = stats[(size_t)K * sb + 1];
        } else {
            denom = 0.0;
            for (int q = 0; q < K; ++q) denom += stats[(size_t)q * sb] + EPS10;
        }
        wk = nk / denom;
        if (p == 0) weights[k] = wk;
        if (p < Dh) {
            const double mx = st[1 + p] / nk, my = st[1 + Dh + p] / nk;
            means[(size_t)k * D + p] = centres[(size_t)k * D + p] + mx;
            means[(size_t)k * D + Dh + p] = centres[(size_t)k * D + Dh + p] + my;
            const double* s2 = st + 1 + D + 3 * p;
            ck[3 * p] = (s2[0] / nk - mx * mx) + reg_covar;
            ck[3 * p + 1] = s2[1] / nk - mx * my;
            ck[3 * p + 2] = (s2[2] / nk - my * my) + reg_covar;
        }
    } else {
        wk = weights[k];
    }
    double ld = 0.0;
    int bad = 0;
    if (p < Dh) {
        const double sxx = ck[3 * p], sxy = ck[3 * p + 1], syy = ck[3 * p + 2];
        // L = [[l11, 0], [l21, l22]] with Sigma = L L^T; U = L^-T
        const bool fail_x = !(sxx > 0.0);
        const double a = 1.0 / sqrt(fail_x ? 1.0 : sxx);
        const double l21 = sxy * a;
        const double t = syy - l21 * l21;
        const bool fail_y = !(t > 0.0);
        const double c = 1.0 / sqrt(fail_y ? 1.0 : t);
        double* U = factors + (size_t)k * 3 * Dh + 3 * p;
        U[0] = a;
        U[1] = -l21 * a * c;
        U[2] = c;
        ld = log(a) + log(c);
        bad = fail_x ? p + 1 : fail_y ? Dh + p + 1 : 0;
    }
    sh_ld[p] = ld;
    sh_bad[p] = bad;
    __syncthreads();
    if (p == 0) {
        double t = 0.0;
        int first = 0;
        for (int q = 0; q < Dh; ++q) {
            t += sh_ld[q];
            const int b = sh_bad[q];
            if (b != 0 && (first == 0 || b < first)) first = b;
        }
        aux[2 * k] = t;
        aux[2 * k + 1] = log(wk);
        info[k] = first;
    }
}

// chunks of frames per component in the M-step: about eight CTAs per SM in all.
static int db_chunks(int K) {
    int c = (8 * 148 + K - 1) / K;
    return c < 1 ? 1 : c > 256 ? 256 : c;
}

struct DbWorkspace {
    double* lse_partial;
    double* partial;
};

static DbWorkspace carve_db(Carver& c, long long N, int K, int D) {
    DbWorkspace w;
    w.lse_partial = c.take<double>((size_t)((N + DB_FT - 1) / DB_FT) + 1);
    w.partial = c.take<double>((size_t)db_chunks(K) * K * db_stats_block(D));
    return w;
}

}  // namespace kw

using namespace kw;

extern "C" size_t kw_gmm_db_stats_len(int K, int D) { return (size_t)K * db_stats_block(D) + 2; }

extern "C" size_t kw_gmm_db_workspace_bytes(int64_t n_frames, int K, int D) {
    Carver c(nullptr);
    carve_db(c, n_frames, K, D);
    return align_up(c.used, 256);
}

// The checks every entry point makes on the shape.
static int db_check_shape(const char* fn, long long N, int K, int D) {
    KW_REQUIRE(N >= 0, "%s: n_frames must be >= 0, got %lld", fn, N);
    KW_REQUIRE(K >= 1, "%s: n_components must be >= 1, got %d", fn, K);
    KW_REQUIRE(D >= 2 && D <= GMM_MAX_DIM && D % 2 == 0,
               "%s: dim must be even with 2 <= dim <= %d, got %d", fn, GMM_MAX_DIM, D);
    return KW_OK;
}

static int db_carve(long long N, int K, int D, void* base, size_t bytes, DbWorkspace& w) {
    Carver c(base);
    w = carve_db(c, N, K, D);
    const size_t need = align_up(c.used, 256);
    if (need > bytes) {
        set_error("GMM workspace too small: need %zu bytes, got %zu", need, bytes);
        return KW_ERR_WORKSPACE;
    }
    return KW_OK;
}

extern "C" int kw_gmm_db_estep(int64_t N, const double* x_dev, int K, int D,
                               const double* means_dev, const double* factors_dev,
                               const double* aux_dev, double* resp_dev, double* stats_dev,
                               double* lse_frame_dev, void* workspace_dev, size_t workspace_bytes,
                               void* stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int rc = db_check_shape("kw_gmm_db_estep", N, K, D);
    if (rc != KW_OK) return rc;
    KW_REQUIRE((N == 0 || (x_dev && resp_dev)) && means_dev && factors_dev && aux_dev &&
                   stats_dev && workspace_dev,
               "kw_gmm_db_estep: a required buffer is NULL");
    DbWorkspace w;
    rc = db_carve(N, K, D, workspace_dev, workspace_bytes, w);
    if (rc != KW_OK) return rc;
    const long long grid = (N + DB_FT - 1) / DB_FT;
    if (grid > 0) {
        const size_t smem = sizeof(double) * (size_t)DB_FT * (D + 1);
        KW_CUDA_CHECK(cudaFuncSetAttribute(gmm_db_estep_kernel,
                                           cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)smem));
        gmm_db_estep_kernel<<<(unsigned)grid, DB_THREADS, smem, st>>>(
            N, resp_pad(N), x_dev, K, D, means_dev, factors_dev, aux_dev, resp_dev,
            w.lse_partial, lse_frame_dev);
        KW_CUDA_CHECK(cudaGetLastError());
    }
    return reduce_fixed(w.lse_partial, grid, (double)N, stats_dev + (size_t)K * db_stats_block(D),
                        st);
}

extern "C" int kw_gmm_db_mstep_accumulate(int64_t N, const double* x_dev, int K, int D,
                                          const double* resp_dev, const double* centres_dev,
                                          double* stats_dev, void* workspace_dev,
                                          size_t workspace_bytes, void* stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int rc = db_check_shape("kw_gmm_db_mstep_accumulate", N, K, D);
    if (rc != KW_OK) return rc;
    KW_REQUIRE((N == 0 || (x_dev && resp_dev)) && centres_dev && stats_dev && workspace_dev,
               "kw_gmm_db_mstep_accumulate: a required buffer is NULL");
    DbWorkspace w;
    rc = db_carve(N, K, D, workspace_dev, workspace_bytes, w);
    if (rc != KW_OK) return rc;
    const int chunks = db_chunks(K);
    const long long fpc = (N + chunks - 1) / chunks;
    gmm_db_mstats_kernel<<<dim3(K, chunks), DB_THREADS, 0, st>>>(
        N, resp_pad(N), x_dev, K, D, resp_dev, centres_dev, w.partial, fpc, RESP_FLOOR);
    KW_CUDA_CHECK(cudaGetLastError());
    gmm_db_reduce_partials_kernel<<<296, 256, 0, st>>>((size_t)K * db_stats_block(D), chunks,
                                                       w.partial, stats_dev);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

extern "C" int kw_gmm_db_mstep_finalize(int K, int D, double reg_covar, int weight_norm,
                                        const double* stats_dev, const double* centres_dev,
                                        double* weights_dev, double* means_dev,
                                        double* covariances_dev, double* factors_dev,
                                        double* aux_dev, int32_t* info_dev, void* stream) {
    int rc = db_check_shape("kw_gmm_db_mstep_finalize", 0, K, D);
    if (rc != KW_OK) return rc;
    KW_REQUIRE(reg_covar >= 0.0, "kw_gmm_db_mstep_finalize: reg_covar must be >= 0, got %g",
               reg_covar);
    KW_REQUIRE(weight_norm == 0 || weight_norm == 1,
               "kw_gmm_db_mstep_finalize: weight_norm must be 0 or 1, got %d", weight_norm);
    KW_REQUIRE(stats_dev && centres_dev && weights_dev && means_dev && covariances_dev &&
                   factors_dev && aux_dev && info_dev,
               "kw_gmm_db_mstep_finalize: a required buffer is NULL");
    gmm_db_finalize_kernel<<<K, DB_FIN_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
        K, D, reg_covar, weight_norm, 1, stats_dev, centres_dev, weights_dev, means_dev,
        covariances_dev, factors_dev, aux_dev, info_dev);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

extern "C" int kw_gmm_db_precision_cholesky(int K, int D, const double* weights_dev,
                                            const double* covariances_dev, double* factors_dev,
                                            double* aux_dev, int32_t* info_dev, void* stream) {
    int rc = db_check_shape("kw_gmm_db_precision_cholesky", 0, K, D);
    if (rc != KW_OK) return rc;
    KW_REQUIRE(weights_dev && covariances_dev && factors_dev && aux_dev && info_dev,
               "kw_gmm_db_precision_cholesky: a required buffer is NULL");
    gmm_db_finalize_kernel<<<K, DB_FIN_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
        K, D, 0.0, 0, 0, nullptr, nullptr, const_cast<double*>(weights_dev), nullptr,
        const_cast<double*>(covariances_dev), factors_dev, aux_dev, info_dev);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

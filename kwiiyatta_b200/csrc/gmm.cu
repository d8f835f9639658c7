// Full-covariance joint-GMM EM, FP64 CUDA-core path (precision = 0), for sm_100a.
//
// Replaces sklearn GaussianMixture.fit as configured at kwiiyatta/converter/gmm.py:9-26
// (formulae: sklearn/mixture/_gaussian_mixture.py _estimate_log_gaussian_prob,
// _estimate_gaussian_parameters, _compute_precision_cholesky; restated in oracle/gmm_ref.py).
//
//   E-step   wlp[n,k] = -1/2 (D log 2pi + || x_n L_k - mu_k L_k ||^2) + log|L_k| + log w_k
//            resp = exp(wlp - logsumexp_k wlp);  sum_n logsumexp -> lower bound
//   M-step   n_k = sum r, m_k = sum r (x - c_k), S_k = sum r (x - c_k)(x - c_k)^T accumulated
//            around the previous means c_k (so the cancellation in S/n - delta delta^T is
//            second order), partials reduced in a fixed order (bitwise reproducible)
//   finalize weights, means, covariances (+reg I), Cholesky, triangular inverse -> L, log|L|.
#include <cfloat>
#include <climits>

#include "common.cuh"

namespace kw {

constexpr int E_FT = 64;   // frames per CTA tile in the E-step
constexpr int E_KC = 16;   // contraction chunk
constexpr int M_FB = 8;    // frames per smem stage in the M-step (static smem < 48 KB)

__host__ __device__ static inline size_t stats_block(int D) { return 1 + (size_t)D + (size_t)D * D; }

// ---------------------------------------------------------------------------------------
// E-step.  CTA = 64 frames x all K components.  256 threads = 16 frame groups (4 frames
// each, interleaved) x 16 column groups (TN contiguous columns each).
// mode 0: write resp + per-CTA sum of logsumexp (and, when lse_frame is not NULL, the logsumexp
// of every frame).  mode 1: hard argmax (np.argmax: first max).
// ---------------------------------------------------------------------------------------
template <int TN>
__global__ void __launch_bounds__(256)
gmm_estep_kernel(long long N, long long Npad, const double* __restrict__ X, int K, int D,
                 const double* __restrict__ prec_chol, const double* __restrict__ aux,
                 double* __restrict__ resp, double* __restrict__ lse_partial, int mode,
                 int32_t* __restrict__ mix_out, double* __restrict__ lse_frame) {
    constexpr int WT = 16 * TN;
    extern __shared__ double sm[];
    const int Dp = (D + E_KC - 1) / E_KC * E_KC;
    const int XS = Dp + 1;
    double* xs = sm;                 // E_FT * XS
    double* ls = xs + E_FT * XS;     // 2 * E_KC * WT
    __shared__ double frame_lse[E_FT];

    const int tid = threadIdx.x;
    const int tr = tid >> 4, tc = tid & 15;
    const long long n0 = (long long)blockIdx.x * E_FT;
    const int nchunks = Dp / E_KC;
    const double LOG2PI = 1.8378770664093453;

    for (int e = tid; e < E_FT * Dp; e += 256) {
        const int f = e / Dp, dd = e - f * Dp;
        const long long n = n0 + f;
        xs[f * XS + dd] = (n < N && dd < D) ? X[n * D + dd] : 0.0;
    }

    double best_v[4];
    int best_k[4];
#pragma unroll
    for (int m = 0; m < 4; ++m) { best_v[m] = -CUDART_INF; best_k[m] = 0; }

    for (int k = 0; k < K; ++k) {
        const double* __restrict__ Lk = prec_chol + (size_t)k * D * D;
        double acc[4][TN];
#pragma unroll
        for (int m = 0; m < 4; ++m)
#pragma unroll
            for (int c = 0; c < TN; ++c) acc[m][c] = 0.0;
        double pre[TN];
        auto prefetch = [&](int dc) {
#pragma unroll
            for (int q = 0; q < TN; ++q) {
                const int e = tid + 256 * q;
                const int dd = e / WT, j = e - dd * WT;
                const int dg = dc * E_KC + dd;
                pre[q] = (dg < D && j < D) ? Lk[(size_t)dg * D + j] : 0.0;
            }
        };
        auto stash = [&](int buf) {
#pragma unroll
            for (int q = 0; q < TN; ++q) ls[buf * E_KC * WT + tid + 256 * q] = pre[q];
        };
        prefetch(0);
        __syncthreads();  // previous k finished reading ls / first pass: xs complete
        stash(0);
        __syncthreads();
        for (int dc = 0; dc < nchunks; ++dc) {
            if (dc + 1 < nchunks) prefetch(dc + 1);
            const double* lb = ls + (dc & 1) * E_KC * WT + tc * TN;
            const double* xb = xs + tr * XS + dc * E_KC;
#pragma unroll
            for (int dd = 0; dd < E_KC; ++dd) {
                double a[4], b[TN];
#pragma unroll
                for (int m = 0; m < 4; ++m) a[m] = xb[(16 * m) * XS + dd];
#pragma unroll
                for (int c = 0; c < TN; ++c) b[c] = lb[dd * WT + c];
#pragma unroll
                for (int m = 0; m < 4; ++m)
#pragma unroll
                    for (int c = 0; c < TN; ++c) acc[m][c] = fma(a[m], b[c], acc[m][c]);
            }
            if (dc + 1 < nchunks) stash((dc + 1) & 1);
            __syncthreads();
        }
        const double* ak = aux + (size_t)k * (D + 2);
        double bk[TN];
#pragma unroll
        for (int c = 0; c < TN; ++c) {
            const int j = tc * TN + c;
            bk[c] = (j < D) ? ak[j] : 0.0;
        }
        const double cst = ak[D] /* log|L| */, lw = ak[D + 1];
#pragma unroll
        for (int m = 0; m < 4; ++m) {
            double q = 0.0;
#pragma unroll
            for (int c = 0; c < TN; ++c) {
                const double y = acc[m][c] - bk[c];
                q = fma(y, y, q);
            }
            q += __shfl_xor_sync(0xffffffffu, q, 8);
            q += __shfl_xor_sync(0xffffffffu, q, 4);
            q += __shfl_xor_sync(0xffffffffu, q, 2);
            q += __shfl_xor_sync(0xffffffffu, q, 1);
            if (tc == 0) {
                const long long n = n0 + tr + 16 * m;
                const double wlp = (-0.5 * ((double)D * LOG2PI + q) + cst) + lw;
                if (mode == 0) {
                    if (n < N) __stcg(resp + (size_t)k * Npad + n, wlp);
                } else if (wlp > best_v[m]) {
                    best_v[m] = wlp;
                    best_k[m] = k;
                }
            }
        }
    }
    if (mode == 1) {
        if (tc == 0) {
#pragma unroll
            for (int m = 0; m < 4; ++m) {
                const long long n = n0 + tr + 16 * m;
                if (n < N) mix_out[n] = best_k[m];
            }
        }
        return;
    }
    __syncthreads();
    // logsumexp over components, one thread per frame (coalesced over the frame index)
    if (tid < E_FT) {
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
        for (int f = 0; f < E_FT; ++f) t += frame_lse[f];
        lse_partial[blockIdx.x] = t;
    }
}

// Sum `n` doubles in a fixed order (single CTA) and write {sum, extra} to out[0], out[1].
__global__ void reduce_fixed_kernel(const double* __restrict__ in, long long n, double extra,
                                    double* __restrict__ out) {
    __shared__ double sh[256];
    double s = 0.0;
    for (long long i = threadIdx.x; i < n; i += 256) s += in[i];
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        out[0] = sh[0];
        out[1] = extra;
    }
}

// ---------------------------------------------------------------------------------------
// M-step sufficient statistics: grid (K, n_chunks, n_tile_pairs).  CTA = one W x W output tile
// (W = 16*TM) of S_k over one chunk of frames; 256 threads, TM x TM accumulators each.
// Frames whose responsibility for this component is <= resp_floor are skipped: the chunk is
// compacted in frame order (deterministic block scan), so the summation order is fixed and
// the work follows the posterior's sparsity.  The diagonal tile CTAs also accumulate
// m_k = sum r (x - c_k) for their rows; tile 0 accumulates n_k = sum r.
// partial layout: [chunk][k][1 + D + D*D].
// ---------------------------------------------------------------------------------------
constexpr int M_SEG = 256;

template <int TM>
__global__ void __launch_bounds__(256)
gmm_mstats_kernel(long long N, long long Npad, const double* __restrict__ X, int K, int D,
                  const double* __restrict__ respT, const double* __restrict__ centres,
                  double* __restrict__ partial, long long frames_per_chunk, int n_tiles,
                  double resp_floor) {
    constexpr int W = 16 * TM;
    constexpr int WS = W + 1;
    constexpr int QCAP = M_SEG + M_FB;
    __shared__ double sa[2][M_FB * WS];
    __shared__ double sb[2][M_FB * WS];
    __shared__ int q_n[QCAP];
    __shared__ double q_r[QCAP];
    __shared__ int warp_cnt[8];
    const int tid = threadIdx.x;
    const int ty = tid >> 4, tx = tid & 15;
    const int lane = tid & 31, warp = tid >> 5;
    const int k = blockIdx.x;
    int bi = 0, bj = 0;
    {
        int t = blockIdx.z;
        for (bi = 0; bi < n_tiles; ++bi) {
            const int row = n_tiles - bi;
            if (t < row) { bj = bi + t; break; }
            t -= row;
        }
    }
    const bool same = (bi == bj);
    const long long n_begin = (long long)blockIdx.y * frames_per_chunk;
    const long long n_end = min(N, n_begin + frames_per_chunk);
    const double* ck = centres + (size_t)k * D;
    const double* rk = respT + (size_t)k * Npad;

    double acc[TM][TM];
    double macc[TM];
    double nacc = 0.0;
#pragma unroll
    for (int a = 0; a < TM; ++a) {
        macc[a] = 0.0;
#pragma unroll
        for (int b = 0; b < TM; ++b) acc[a][b] = 0.0;
    }

    constexpr int PER = (M_FB * W + 255) / 256;
    double pa[PER], pb[PER];
    auto prefetch = [&](int q0) {   // batch of M_FB queue entries starting at q0
#pragma unroll
        for (int q = 0; q < PER; ++q) {
            const int e = tid + 256 * q;
            const int f = e / W, c = e - f * W;
            double va = 0.0, vb = 0.0;
            if (e < M_FB * W) {
                const double r = q_r[q0 + f];
                const long long n = n_begin + q_n[q0 + f];
                const int ci = bi * W + c, cj = bj * W + c;
                const double xi = (ci < D) ? X[n * D + ci] - ck[ci] : 0.0;
                va = r * xi;
                vb = same ? xi : ((cj < D) ? X[n * D + cj] - ck[cj] : 0.0);
            }
            pa[q] = va;
            pb[q] = vb;
        }
    };
    auto stash = [&](int buf) {
#pragma unroll
        for (int q = 0; q < PER; ++q) {
            const int e = tid + 256 * q;
            if (e < M_FB * W) {
                const int f = e / W, c = e - f * W;
                sa[buf][f * WS + c] = pa[q];
                sb[buf][f * WS + c] = pb[q];
            }
        }
    };
    // consume n_batches full batches from the front of the queue
    auto process = [&](int n_batches) {
        if (n_batches <= 0) return;
        prefetch(0);
        stash(0);
        __syncthreads();
        int buf = 0;
        for (int b = 0; b < n_batches; ++b) {
            const bool more = b + 1 < n_batches;
            if (more) prefetch((b + 1) * M_FB);
            const double* a_base = sa[buf] + ty * TM;
            const double* b_base = sb[buf] + tx * TM;
#pragma unroll
            for (int f = 0; f < M_FB; ++f) {
                double a[TM], bb[TM];
#pragma unroll
                for (int q = 0; q < TM; ++q) a[q] = a_base[f * WS + q];
#pragma unroll
                for (int q = 0; q < TM; ++q) bb[q] = b_base[f * WS + q];
#pragma unroll
                for (int p = 0; p < TM; ++p)
#pragma unroll
                    for (int q = 0; q < TM; ++q) acc[p][q] = fma(a[p], bb[q], acc[p][q]);
                if (same && tx == 0) {
#pragma unroll
                    for (int p = 0; p < TM; ++p) macc[p] += a[p];
                }
                if (tid == 0) nacc += q_r[b * M_FB + f];
            }
            if (more) stash(buf ^ 1);
            __syncthreads();
            buf ^= 1;
        }
    };

    int qcount = 0;
    for (long long seg = n_begin; seg < n_end; seg += M_SEG) {
        const long long n = seg + tid;
        const double r = (n < n_end) ? rk[n] : 0.0;
        const bool keep = r > resp_floor;
        const unsigned ballot = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) warp_cnt[warp] = __popc(ballot);
        __syncthreads();
        int before = 0, total = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) {
            const int c = warp_cnt[w];
            if (w < warp) before += c;
            total += c;
        }
        if (keep) {
            const int pos = qcount + before + __popc(ballot & ((1u << lane) - 1u));
            q_n[pos] = (int)(n - n_begin);
            q_r[pos] = r;
        }
        qcount += total;
        __syncthreads();
        const int nb = qcount / M_FB;
        process(nb);
        const int rem = qcount - nb * M_FB;
        int tn = 0;
        double tr = 0.0;
        if (nb > 0 && tid < rem) { tn = q_n[nb * M_FB + tid]; tr = q_r[nb * M_FB + tid]; }
        __syncthreads();
        if (nb > 0 && tid < rem) { q_n[tid] = tn; q_r[tid] = tr; }
        qcount = rem;
        __syncthreads();
    }
    if (qcount > 0) {
        if (tid >= qcount && tid < M_FB) { q_n[tid] = 0; q_r[tid] = 0.0; }
        __syncthreads();
        process(1);
    }

    double* out = partial + ((size_t)blockIdx.y * K + k) * stats_block(D);
    if (blockIdx.z == 0 && tid == 0) out[0] = nacc;
    if (same && tx == 0) {
#pragma unroll
        for (int p = 0; p < TM; ++p) {
            const int i = bi * W + ty * TM + p;
            if (i < D) out[1 + i] = macc[p];
        }
    }
    double* so = out + 1 + D;
#pragma unroll
    for (int p = 0; p < TM; ++p) {
        const int i = bi * W + ty * TM + p;
        if (i >= D) continue;
#pragma unroll
        for (int q = 0; q < TM; ++q) {
            const int j = bj * W + tx * TM + q;
            if (j >= D) continue;
            so[(size_t)i * D + j] = acc[p][q];
            if (!same) so[(size_t)j * D + i] = acc[p][q];
        }
    }
}

// stats[k] = sum over chunks (fixed order) of the partials.
__global__ void gmm_reduce_partials_kernel(int K, int D, int chunks,
                                           const double* __restrict__ partial,
                                           double* __restrict__ stats) {
    const size_t sb = stats_block(D);
    const size_t total = (size_t)K * sb;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total;
         e += (size_t)gridDim.x * blockDim.x) {
        double s = 0.0;
        for (int c = 0; c < chunks; ++c) s += partial[(size_t)c * total + e];
        stats[e] = s;
    }
}

// ---------------------------------------------------------------------------------------
// Finalize: one CTA (512 threads) per component.  from_stats = 1: parameters from sufficient
// statistics; from_stats = 0: only the precision Cholesky of given covariances (weights/means
// given).  Everything stays in shared memory: covariance -> Cholesky factor L in the lower
// triangle -> Z = L^-1 stored transposed in the strict upper triangle (= the precision
// Cholesky factor sklearn keeps).  Both factorisations are blocked by FIN_NB columns so the
// bulk of the flops are register-tiled panel products and the number of block-wide barriers
// is ~2 per column instead of 3 plus a serial triangular sweep.
// Dynamic smem: D * S doubles (S = D | 1), FIN_NB + 1 doubles per column of scratch (for at
// least two columns: the diagonal block also keeps its 1 / L[c][c] at scratch offset 2 FIN_NB,
// past the end of a one-column scratch), 3 D doubles of diagonals / means.
// ---------------------------------------------------------------------------------------
constexpr int FIN_NB = 16;
constexpr int FIN_THREADS = 512;

__host__ __device__ inline size_t finalize_scratch(int D) {
    return (size_t)(D > 2 ? D : 2) * (FIN_NB + 1);
}
static size_t finalize_smem_bytes(int D) {
    const size_t S = (size_t)D | 1;
    return sizeof(double) * ((size_t)D * S + finalize_scratch(D) + 3 * (size_t)D);
}

__global__ void __launch_bounds__(FIN_THREADS)
gmm_finalize_kernel(int K, int D, double reg_covar, int weight_norm, int from_stats,
                    const double* __restrict__ stats, const double* __restrict__ centres,
                    double* __restrict__ weights, double* __restrict__ means,
                    double* __restrict__ covariances, double* __restrict__ prec_chol,
                    double* __restrict__ aux, int32_t* __restrict__ info) {
    extern __shared__ double A[];
    const int S = D | 1;
    double* T = A + (size_t)D * S;            // [column][FIN_NB + 1] scratch of the inverse
    double* dg = T + finalize_scratch(D);     // L[j][j]
    double* zd = dg + D;                      // 1 / L[j][j]
    double* dm = zd + D;                      // first moments / n_k
    __shared__ int sh_fail;
    __shared__ double sh_red[FIN_THREADS / 32];
    const int k = blockIdx.x, tid = threadIdx.x;
    double* cov = covariances + (size_t)k * D * D;
    double* mu = means + (size_t)k * D;
    double wk;
    if (from_stats) {
        const size_t sb = stats_block(D);
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
        const double* ck = centres + (size_t)k * D;
        for (int dd = tid; dd < D; dd += FIN_THREADS) {
            const double m = st[1 + dd] / nk;
            dm[dd] = m;
            mu[dd] = ck[dd] + m;
        }
        if (tid == 0) weights[k] = wk;
        __syncthreads();
        for (int i = tid >> 5; i < D; i += FIN_THREADS / 32) {
            const double di = dm[i];
            for (int j = tid & 31; j < D; j += 32) {
                double c = st[1 + D + (size_t)i * D + j] / nk - di * dm[j];
                if (i == j) c += reg_covar;
                cov[(size_t)i * D + j] = c;
                A[i * S + j] = c;
            }
        }
    } else {
        wk = weights[k];
        for (int i = tid >> 5; i < D; i += FIN_THREADS / 32)
            for (int j = tid & 31; j < D; j += 32) A[i * S + j] = cov[(size_t)i * D + j];
    }
    if (tid == 0) sh_fail = 0;
    __syncthreads();

    // ---- Cholesky, left-looking by panels of FIN_NB columns --------------------------------
    // Per element the products are subtracted in ascending column order (the arithmetic of an
    // unblocked left-looking sweep).
    for (int J = 0; J < D; J += FIN_NB) {
        const int nb = min(FIN_NB, D - J);
        if (J > 0) {
            // panel -= L[:, :J] L[J:J+nb, :J]^T; a thread owns 2 rows x 4 columns
            const int R = D - J, Rh = (R + 1) >> 1;
            for (int u = tid; u < Rh * 4; u += FIN_THREADS) {
                const int cg = u / Rh, ip = u - cg * Rh;
                const int c0 = 4 * cg;
                if (c0 >= nb) continue;
                const int i0 = J + ip, i1 = i0 + Rh;
                const bool two = i1 < D;
                const double* r0 = A + i0 * S;
                const double* r1 = A + (two ? i1 : i0) * S;
                const double* q0 = A + (J + c0) * S;
                const double* q1 = A + (J + min(c0 + 1, nb - 1)) * S;
                const double* q2 = A + (J + min(c0 + 2, nb - 1)) * S;
                const double* q3 = A + (J + min(c0 + 3, nb - 1)) * S;
                double a00 = r0[J + c0], a01 = r0[J + min(c0 + 1, nb - 1)],
                       a02 = r0[J + min(c0 + 2, nb - 1)], a03 = r0[J + min(c0 + 3, nb - 1)];
                double a10 = r1[J + c0], a11 = r1[J + min(c0 + 1, nb - 1)],
                       a12 = r1[J + min(c0 + 2, nb - 1)], a13 = r1[J + min(c0 + 3, nb - 1)];
#pragma unroll 8
                for (int p = 0; p < J; ++p) {
                    const double l0 = -r0[p], l1 = -r1[p];
                    const double b0 = q0[p], b1 = q1[p], b2 = q2[p], b3 = q3[p];
                    a00 = fma(l0, b0, a00); a01 = fma(l0, b1, a01);
                    a02 = fma(l0, b2, a02); a03 = fma(l0, b3, a03);
                    a10 = fma(l1, b0, a10); a11 = fma(l1, b1, a11);
                    a12 = fma(l1, b2, a12); a13 = fma(l1, b3, a13);
                }
                double* w0 = A + i0 * S + J + c0;
                double* w1 = A + i1 * S + J + c0;
                w0[0] = a00;
                if (c0 + 1 < nb) w0[1] = a01;
                if (c0 + 2 < nb) w0[2] = a02;
                if (c0 + 3 < nb) w0[3] = a03;
                if (two) {
                    w1[0] = a10;
                    if (c0 + 1 < nb) w1[1] = a11;
                    if (c0 + 2 < nb) w1[2] = a12;
                    if (c0 + 3 < nb) w1[3] = a13;
                }
            }
            __syncthreads();
        }
        // Inside the panel, two barriers instead of one per column.  Per element the products are
        // still subtracted in ascending column order.  (Measured with clocks in block 0 before
        // commit 3a91ef5: of the Cholesky's 136k clk the left-looking panel updates take 69k -- few
        // warps are active in the late panels and the dot products wait for shared memory -- the
        // diagonal blocks 80k, 550 clk per pivot in one warp, the rows below 22k.)
        // (a) the nb x nb diagonal block in ONE warp: lane r keeps row r in registers, the pivot
        //     column travels through a small shared-memory line.
        if (tid < 32) {
            // branch-free straight-line code (the 16 row values are named scalars: as an indexed
            // array the compiler kept them in local memory), so that the scheduler can run the next
            // pivot's rsqrt under the rest of this column's updates; rows past nb act as identity
            // rows.  Lane r keeps row r of the block; L[q][c] reaches the other lanes by shuffle.
            static_assert(FIN_NB == 16, "the diagonal-block code below is written out for 16 columns");
            const int lane = tid;
            double a0 = (lane < nb && 0 <= lane) ? A[(J + lane) * S + J + 0] : ((lane >= nb && lane == 0) ? 1.0 : 0.0);
            double a1 = (lane < nb && 1 <= lane) ? A[(J + lane) * S + J + 1] : ((lane >= nb && lane == 1) ? 1.0 : 0.0);
            double a2 = (lane < nb && 2 <= lane) ? A[(J + lane) * S + J + 2] : ((lane >= nb && lane == 2) ? 1.0 : 0.0);
            double a3 = (lane < nb && 3 <= lane) ? A[(J + lane) * S + J + 3] : ((lane >= nb && lane == 3) ? 1.0 : 0.0);
            double a4 = (lane < nb && 4 <= lane) ? A[(J + lane) * S + J + 4] : ((lane >= nb && lane == 4) ? 1.0 : 0.0);
            double a5 = (lane < nb && 5 <= lane) ? A[(J + lane) * S + J + 5] : ((lane >= nb && lane == 5) ? 1.0 : 0.0);
            double a6 = (lane < nb && 6 <= lane) ? A[(J + lane) * S + J + 6] : ((lane >= nb && lane == 6) ? 1.0 : 0.0);
            double a7 = (lane < nb && 7 <= lane) ? A[(J + lane) * S + J + 7] : ((lane >= nb && lane == 7) ? 1.0 : 0.0);
            double a8 = (lane < nb && 8 <= lane) ? A[(J + lane) * S + J + 8] : ((lane >= nb && lane == 8) ? 1.0 : 0.0);
            double a9 = (lane < nb && 9 <= lane) ? A[(J + lane) * S + J + 9] : ((lane >= nb && lane == 9) ? 1.0 : 0.0);
            double a10 = (lane < nb && 10 <= lane) ? A[(J + lane) * S + J + 10] : ((lane >= nb && lane == 10) ? 1.0 : 0.0);
            double a11 = (lane < nb && 11 <= lane) ? A[(J + lane) * S + J + 11] : ((lane >= nb && lane == 11) ? 1.0 : 0.0);
            double a12 = (lane < nb && 12 <= lane) ? A[(J + lane) * S + J + 12] : ((lane >= nb && lane == 12) ? 1.0 : 0.0);
            double a13 = (lane < nb && 13 <= lane) ? A[(J + lane) * S + J + 13] : ((lane >= nb && lane == 13) ? 1.0 : 0.0);
            double a14 = (lane < nb && 14 <= lane) ? A[(J + lane) * S + J + 14] : ((lane >= nb && lane == 14) ? 1.0 : 0.0);
            double a15 = (lane < nb && 15 <= lane) ? A[(J + lane) * S + J + 15] : ((lane >= nb && lane == 15) ? 1.0 : 0.0);
            unsigned bad = 0u;
            double my_dg = 0.0, my_rinv = 0.0;
#define FIN_UPD(q)                                                        \
    {                                                                     \
        const double lq = __shfl_sync(0xffffffffu, l_rc, q);              \
        if (lane >= q) a##q = fma(l_rc, -lq, a##q);                       \
    }
#define FIN_STEP(c, UPDS)                                                 \
    {                                                                     \
        double s = __shfl_sync(0xffffffffu, a##c, c);                     \
        const bool fail = !(s > 0.0);                                     \
        bad |= fail ? (1u << c) : 0u;                                     \
        s = fail ? 1.0 : s;                                               \
        const double rinv = rsqrt(s);                                     \
        if (lane == c) {                                                  \
            my_dg = s * rinv;                                             \
            my_rinv = rinv;                                               \
        }                                                                 \
        const double l_rc = a##c * rinv; /* L[r][c] for the lanes r > c */ \
        UPDS                                                              \
        if (lane > c) a##c = l_rc;                                        \
    }
            FIN_STEP(0, FIN_UPD(1) FIN_UPD(2) FIN_UPD(3) FIN_UPD(4) FIN_UPD(5) FIN_UPD(6) FIN_UPD(7) FIN_UPD(8) FIN_UPD(9) FIN_UPD(10) FIN_UPD(11) FIN_UPD(12) FIN_UPD(13) FIN_UPD(14) FIN_UPD(15))
            FIN_STEP(1, FIN_UPD(2) FIN_UPD(3) FIN_UPD(4) FIN_UPD(5) FIN_UPD(6) FIN_UPD(7) FIN_UPD(8) FIN_UPD(9) FIN_UPD(10) FIN_UPD(11) FIN_UPD(12) FIN_UPD(13) FIN_UPD(14) FIN_UPD(15))
            FIN_STEP(2, FIN_UPD(3) FIN_UPD(4) FIN_UPD(5) FIN_UPD(6) FIN_UPD(7) FIN_UPD(8) FIN_UPD(9) FIN_UPD(10) FIN_UPD(11) FIN_UPD(12) FIN_UPD(13) FIN_UPD(14) FIN_UPD(15))
            FIN_STEP(3, FIN_UPD(4) FIN_UPD(5) FIN_UPD(6) FIN_UPD(7) FIN_UPD(8) FIN_UPD(9) FIN_UPD(10) FIN_UPD(11) FIN_UPD(12) FIN_UPD(13) FIN_UPD(14) FIN_UPD(15))
            FIN_STEP(4, FIN_UPD(5) FIN_UPD(6) FIN_UPD(7) FIN_UPD(8) FIN_UPD(9) FIN_UPD(10) FIN_UPD(11) FIN_UPD(12) FIN_UPD(13) FIN_UPD(14) FIN_UPD(15))
            FIN_STEP(5, FIN_UPD(6) FIN_UPD(7) FIN_UPD(8) FIN_UPD(9) FIN_UPD(10) FIN_UPD(11) FIN_UPD(12) FIN_UPD(13) FIN_UPD(14) FIN_UPD(15))
            FIN_STEP(6, FIN_UPD(7) FIN_UPD(8) FIN_UPD(9) FIN_UPD(10) FIN_UPD(11) FIN_UPD(12) FIN_UPD(13) FIN_UPD(14) FIN_UPD(15))
            FIN_STEP(7, FIN_UPD(8) FIN_UPD(9) FIN_UPD(10) FIN_UPD(11) FIN_UPD(12) FIN_UPD(13) FIN_UPD(14) FIN_UPD(15))
            FIN_STEP(8, FIN_UPD(9) FIN_UPD(10) FIN_UPD(11) FIN_UPD(12) FIN_UPD(13) FIN_UPD(14) FIN_UPD(15))
            FIN_STEP(9, FIN_UPD(10) FIN_UPD(11) FIN_UPD(12) FIN_UPD(13) FIN_UPD(14) FIN_UPD(15))
            FIN_STEP(10, FIN_UPD(11) FIN_UPD(12) FIN_UPD(13) FIN_UPD(14) FIN_UPD(15))
            FIN_STEP(11, FIN_UPD(12) FIN_UPD(13) FIN_UPD(14) FIN_UPD(15))
            FIN_STEP(12, FIN_UPD(13) FIN_UPD(14) FIN_UPD(15))
            FIN_STEP(13, FIN_UPD(14) FIN_UPD(15))
            FIN_STEP(14, FIN_UPD(15))
            FIN_STEP(15, )
#undef FIN_STEP
#undef FIN_UPD
            if (lane < nb) {
                dg[J + lane] = my_dg;
                T[FIN_NB * 2 + lane] = my_rinv;              // 1 / L[c][c] for the rows below
            }
            bad &= (1u << nb) - 1u;
            if (lane == 0 && bad != 0u && sh_fail == 0) sh_fail = J + __ffs(bad);
            // L values below the diagonal back into the block (the diagonal keeps its pre-pivot
            // value, as before)
            if (lane < nb && 0 < lane) A[(J + lane) * S + J + 0] = a0;
            if (lane < nb && 1 < lane) A[(J + lane) * S + J + 1] = a1;
            if (lane < nb && 2 < lane) A[(J + lane) * S + J + 2] = a2;
            if (lane < nb && 3 < lane) A[(J + lane) * S + J + 3] = a3;
            if (lane < nb && 4 < lane) A[(J + lane) * S + J + 4] = a4;
            if (lane < nb && 5 < lane) A[(J + lane) * S + J + 5] = a5;
            if (lane < nb && 6 < lane) A[(J + lane) * S + J + 6] = a6;
            if (lane < nb && 7 < lane) A[(J + lane) * S + J + 7] = a7;
            if (lane < nb && 8 < lane) A[(J + lane) * S + J + 8] = a8;
            if (lane < nb && 9 < lane) A[(J + lane) * S + J + 9] = a9;
            if (lane < nb && 10 < lane) A[(J + lane) * S + J + 10] = a10;
            if (lane < nb && 11 < lane) A[(J + lane) * S + J + 11] = a11;
            if (lane < nb && 12 < lane) A[(J + lane) * S + J + 12] = a12;
            if (lane < nb && 13 < lane) A[(J + lane) * S + J + 13] = a13;
            if (lane < nb && 14 < lane) A[(J + lane) * S + J + 14] = a14;
        }
        __syncthreads();
        // (b) the rows below the block, one thread per row: forward substitution against the block
        for (int i = J + nb + tid; i < D; i += FIN_THREADS) {
            double x[FIN_NB];
#pragma unroll
            for (int c = 0; c < FIN_NB; ++c) {
                if (c < nb) {
                    double v = A[i * S + J + c];
#pragma unroll
                    for (int q = 0; q < c; ++q) v = fma(x[q], -A[(J + c) * S + J + q], v);
                    x[c] = v * T[FIN_NB * 2 + c];
                }
            }
#pragma unroll
            for (int c = 0; c < FIN_NB; ++c)
                if (c < nb) A[i * S + J + c] = x[c];
        }
        __syncthreads();
    }
    // (A[j][j] still holds the pre-pivot value; the diagonal of L lives in dg)
    for (int j = tid; j < D; j += FIN_THREADS) zd[j] = 1.0 / dg[j];
    __syncthreads();

    // ---- Z = L^-1 by block rows; Z^T goes to the strict upper triangle: A[c][r] = Z[r][c] ----
    // diagonal blocks: one thread per column, forward substitution in registers
    {
        const int nblk = (D + FIN_NB - 1) / FIN_NB;
        if (tid < nblk * FIN_NB) {
            const int I = tid / FIN_NB, c = tid - I * FIN_NB, base = I * FIN_NB;
            const int nb = min(FIN_NB, D - base);
            if (c < nb) {
                double z[FIN_NB];
#pragma unroll
                for (int r = 0; r < FIN_NB; ++r) z[r] = 0.0;
#pragma unroll
                for (int r = 0; r < FIN_NB; ++r) {
                    if (r == c) z[r] = zd[base + r];
                    if (r > c && r < nb) {
                        double acc = 0.0;
#pragma unroll
                        for (int q = 0; q < FIN_NB; ++q)
                            if (q < r) acc = fma(A[(base + r) * S + base + q], z[q], acc);
                        z[r] = -acc * zd[base + r];
                        A[(base + c) * S + base + r] = z[r];
                    }
                }
            }
        }
    }
    __syncthreads();
    for (int I0 = FIN_NB; I0 < D; I0 += FIN_NB) {
        const int nb = min(FIN_NB, D - I0);
        // T[r][c] = sum_{p = c}^{I0 - 1} L[I0 + r][p] Z[p][c];  thread: rows (rp, rp + 8),
        // columns (c, c + 1)
        for (int u = tid; u < 8 * (I0 / 2); u += FIN_THREADS) {
            const int rp = u & 7, c = (u >> 3) * 2;
            const int ra = min(rp, nb - 1), rb = min(rp + 8, nb - 1);
            const double* la = A + (I0 + ra) * S;
            const double* lb = A + (I0 + rb) * S;
            const double* z0 = A + c * S;
            const double* z1 = A + (c + 1) * S;
            // p = c and p = c + 1 by hand (diagonal terms of Z)
            double t00 = la[c] * zd[c], t10 = lb[c] * zd[c];
            t00 = fma(la[c + 1], z0[c + 1], t00);
            t10 = fma(lb[c + 1], z0[c + 1], t10);
            double t01 = la[c + 1] * zd[c + 1], t11 = lb[c + 1] * zd[c + 1];
#pragma unroll 8
            for (int p = c + 2; p < I0; ++p) {
                const double xa = la[p], xb = lb[p], y0 = z0[p], y1 = z1[p];
                t00 = fma(xa, y0, t00); t01 = fma(xa, y1, t01);
                t10 = fma(xb, y0, t10); t11 = fma(xb, y1, t11);
            }
            T[c * (FIN_NB + 1) + rp] = t00;
            T[(c + 1) * (FIN_NB + 1) + rp] = t01;
            T[c * (FIN_NB + 1) + rp + 8] = t10;
            T[(c + 1) * (FIN_NB + 1) + rp + 8] = t11;
        }
        __syncthreads();
        // Z[I0 + r][c] = - sum_{q <= r} Zdiag[r][q] T[q][c]
        for (int u = tid; u < FIN_NB * I0; u += FIN_THREADS) {
            const int r = u & (FIN_NB - 1), c = u >> 4;
            if (r < nb) {
                const double* tc = T + c * (FIN_NB + 1);
                double acc = zd[I0 + r] * tc[r];
                for (int q = 0; q < r; ++q) acc = fma(A[(I0 + q) * S + I0 + r], tc[q], acc);
                A[c * S + I0 + r] = -acc;
            }
        }
        __syncthreads();
    }
    // prec_chol (upper) = Z^T; diagonal 1 / L[j][j]
    double* pc = prec_chol + (size_t)k * D * D;
    for (int r = tid >> 5; r < D; r += FIN_THREADS / 32)
        for (int c = tid & 31; c < D; c += 32) {
            double v = 0.0;
            if (c > r) v = A[r * S + c];
            else if (c == r) v = zd[r];
            pc[(size_t)r * D + c] = v;
        }
    double ld = 0.0;
    for (int j = tid; j < D; j += FIN_THREADS) ld += log(zd[j]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ld += __shfl_xor_sync(0xffffffffu, ld, o);
    if ((tid & 31) == 0) sh_red[tid >> 5] = ld;
    __syncthreads();
    double* ak = aux + (size_t)k * (D + 2);
    if (tid < D) {
        const int j = tid;
        double b = 0.0;
        for (int dd = 0; dd < j; ++dd) b = fma(mu[dd], A[dd * S + j], b);
        b = fma(mu[j], zd[j], b);
        ak[j] = b;
    }
    if (tid == 0) {
        double t = 0.0;
        for (int w = 0; w < FIN_THREADS / 32; ++w) t += sh_red[w];
        ak[D] = t;
        ak[D + 1] = log(wk);
        info[k] = sh_fail;
    }
}

static int m_chunks(int K) {
    int c = (4 * 148 + K - 1) / K;
    if (c < 1) c = 1;
    if (c > 64) c = 64;
    return c;
}

long long resp_pad(long long n) { return (n + 127) / 128 * 128; }

GmmWorkspace carve_gmm(Carver& c, long long N, int K, int D, int precision, GmmUse use) {
    GmmWorkspace w = {};
    if (use == GmmUse::Fit || (use == GmmUse::Posterior && precision == 0))
        w.lse_partial = c.take<double>((size_t)((N + E_FT - 1) / E_FT) + 1);
    if (use == GmmUse::Fit) w.partial = c.take<double>((size_t)m_chunks(K) * K * stats_block(D));
    if (precision == 1) {
        w.tc = carve_tc(c, N, K, D);
        w.lse_partial = w.tc.lse_partial;
    }
    return w;
}

// Columns per thread of the FP64 E-step (TN) and M-step (TM) kernels at dimension D.
static int fp64_class(int D) { return D <= 16 ? 1 : D <= 32 ? 2 : D <= 48 ? 3 : D <= 80 ? 5 : 9; }

// gmm_estep_kernel: mode 0 writes resp, lse_partial and lse_frame; mode 1 the labels.
static int estep_fp64(long long N, const double* X, int K, int D, const double* pc,
                      const double* aux, double* resp, double* lse_partial, int mode,
                      int32_t* labels, cudaStream_t st, double* lse_frame) {
    static_assert(GMM_MAX_DIM <= 16 * 9, "TN = 9 covers GMM_MAX_DIM columns");
    const int TN = fp64_class(D);
    auto kern = TN == 9   ? gmm_estep_kernel<9>
                : TN == 5 ? gmm_estep_kernel<5>
                : TN == 3 ? gmm_estep_kernel<3>
                : TN == 1 ? gmm_estep_kernel<1>
                          : gmm_estep_kernel<2>;
    const int Dp = (D + E_KC - 1) / E_KC * E_KC;
    const size_t smem = sizeof(double) * ((size_t)E_FT * (Dp + 1) + 2 * E_KC * 16 * TN);
    KW_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem));
    const long long grid = (N + E_FT - 1) / E_FT;
    kern<<<(unsigned)grid, 256, smem, st>>>(N, resp_pad(N), X, K, D, pc, aux, resp, lse_partial,
                                            mode, labels, lse_frame);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

int estep_posterior(long long N, const double* X, int K, int D, const double* means,
                    const double* pc, const double* aux, int precision, const GmmWorkspace& w,
                    const Posterior& out, cudaStream_t st) {
    long long n_partials = (N + E_FT - 1) / E_FT;
    const int rc =
        precision == 1
            ? estep_tc_posterior(N, K, D, means, pc, aux, w.tc, out, n_partials, st)
            : estep_fp64(N, X, K, D, pc, aux, out.resp, w.lse_partial, 0, nullptr, st,
                         out.lse_frame);
    if (rc != KW_OK || out.total == nullptr) return rc;
    return reduce_fixed(w.lse_partial, n_partials, (double)N, out.total, st);
}

int reduce_fixed(const double* in, long long n, double extra, double* out, cudaStream_t st) {
    reduce_fixed_kernel<<<1, 256, 0, st>>>(in, n, extra, out);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

int estep_labels(long long N, const double* X, int K, int D, const double* means,
                 const double* pc, const double* aux, int precision, const GmmWorkspace& w,
                 int32_t* labels, cudaStream_t st) {
    if (precision == 1) return estep_tc_labels(N, X, K, D, means, pc, aux, w.tc, labels, st);
    return estep_fp64(N, X, K, D, pc, aux, nullptr, nullptr, 1, labels, st, nullptr);
}

static int mstats_fp64(long long N, const double* X, int K, int D, const double* resp,
                       const double* centres, double* partial, double* stats, double resp_floor,
                       cudaStream_t st) {
    const int TM = fp64_class(D);
    auto kern = TM == 9   ? gmm_mstats_kernel<9>
                : TM == 5 ? gmm_mstats_kernel<5>
                : TM == 3 ? gmm_mstats_kernel<3>
                : TM == 1 ? gmm_mstats_kernel<1>
                          : gmm_mstats_kernel<2>;
    const int chunks = m_chunks(K);
    const int n_tiles = (D + 16 * TM - 1) / (16 * TM);
    long long fpc = (N + chunks - 1) / chunks;
    fpc = (fpc + M_SEG - 1) / M_SEG * M_SEG;
    kern<<<dim3(K, chunks, n_tiles * (n_tiles + 1) / 2), 256, 0, st>>>(
        N, resp_pad(N), X, K, D, resp, centres, partial, fpc, n_tiles, resp_floor);
    KW_CUDA_CHECK(cudaGetLastError());
    gmm_reduce_partials_kernel<<<296, 256, 0, st>>>(K, D, chunks, partial, stats);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

int finalize_launch(int K, int D, double reg_covar, int weight_norm, int from_stats,
                    const double* stats, const double* centres, double* weights, double* means,
                    double* cov, double* pc, double* aux, int32_t* info, cudaStream_t st) {
    if (D > 160) {
        set_error("dim %d > 160 is not supported by the finalize kernel", D);
        return KW_ERR_UNSUPPORTED;
    }
    const size_t smem = finalize_smem_bytes(D);
    KW_CUDA_CHECK(cudaFuncSetAttribute(gmm_finalize_kernel,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    gmm_finalize_kernel<<<K, FIN_THREADS, smem, st>>>(K, D, reg_covar, weight_norm, from_stats, stats,
                                              centres, weights, means, cov, pc, aux, info);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

}  // namespace kw

using namespace kw;

extern "C" size_t kw_gmm_stats_len(int K, int D) { return (size_t)K * stats_block(D) + 2; }

extern "C" size_t kw_gmm_resp_len(int64_t n_frames, int K) { return (size_t)K * (size_t)resp_pad(n_frames); }

extern "C" size_t kw_gmm_workspace_bytes(int64_t n_frames, int K, int D, int precision) {
    Carver c(nullptr);
    carve_gmm(c, n_frames, K, D, precision, GmmUse::Fit);
    return align_up(c.used, 256);
}

static int dim_unsupported(const char* fn, int D) {
    set_error("%s: dim %d > %d is not supported by the E-step and tensor-core kernels", fn, D,
              GMM_MAX_DIM);
    return KW_ERR_UNSUPPORTED;
}

// The layout of kw_gmm_workspace_bytes over the caller's workspace.
static int carve_fit(long long N, int K, int D, int precision, void* base, size_t bytes,
                     GmmWorkspace& w) {
    Carver c(base);
    w = carve_gmm(c, N, K, D, precision, GmmUse::Fit);
    const size_t need = align_up(c.used, 256);
    if (need > bytes) {
        set_error("GMM workspace too small: need %zu bytes, got %zu", need, bytes);
        return KW_ERR_WORKSPACE;
    }
    return KW_OK;
}

extern "C" int kw_gmm_estep(int64_t N, const double* x_dev, int K, int D, const double* means_dev,
                            const double* prec_chol_dev, const double* aux_dev, double* resp_dev,
                            double* stats_dev, int precision, int resp_form,
                            void* workspace_dev, size_t workspace_bytes, void* stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    KW_REQUIRE(N > 0 && K > 0 && D > 0, "kw_gmm_estep: N, K, D must be positive");
    KW_REQUIRE(precision == 0 || precision == 1, "GMM precision must be 0 (fp64) or 1 (tensor)");
    KW_REQUIRE(resp_form == 0 || resp_form == 1, "resp_form must be 0 or 1");
    if (D > GMM_MAX_DIM) return dim_unsupported("kw_gmm_estep", D);
    if (precision == 1 && resp_form == 1 && K > TC_RESP_FORM1_MAX_K) {
        set_error("resp_form 1 supports at most %d components, got %d", TC_RESP_FORM1_MAX_K, K);
        return KW_ERR_UNSUPPORTED;
    }
    GmmWorkspace w;
    int rc = carve_fit(N, K, D, precision, workspace_dev, workspace_bytes, w);
    if (rc != KW_OK) return rc;
    Posterior out;
    out.resp = resp_dev;
    out.total = stats_dev + (size_t)K * stats_block(D);
    out.resp_form = resp_form;
    return estep_posterior(N, x_dev, K, D, means_dev, prec_chol_dev, aux_dev, precision, w, out,
                           st);
}

extern "C" int kw_gmm_normalize_resp(int64_t N, int K, int D, double* resp_dev,
                                     void* workspace_dev, size_t workspace_bytes, void* stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    KW_REQUIRE(N > 0 && K > 0 && D > 0, "kw_gmm_normalize_resp: N, K, D must be positive");
    if (D > GMM_MAX_DIM) return dim_unsupported("kw_gmm_normalize_resp", D);
    GmmWorkspace w;
    int rc = carve_fit(N, K, D, 1, workspace_dev, workspace_bytes, w);
    if (rc != KW_OK) return rc;
    return normalize_resp_tc(N, K, resp_dev, w.tc, st);
}

extern "C" int kw_gmm_hard_labels(int64_t N, const double* x_dev, int K, int D,
                                  const double* means_dev, const double* prec_chol_dev,
                                  const double* aux_dev, int32_t* labels_dev, int precision,
                                  void* workspace_dev, size_t workspace_bytes, void* stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    KW_REQUIRE(N > 0 && K > 0 && D > 0, "kw_gmm_hard_labels: N, K, D must be positive");
    KW_REQUIRE(precision == 0 || precision == 1, "GMM precision must be 0 (fp64) or 1 (tensor)");
    if (D > GMM_MAX_DIM) return dim_unsupported("kw_gmm_hard_labels", D);
    GmmWorkspace w;
    int rc = carve_fit(N, K, D, precision, workspace_dev, workspace_bytes, w);
    if (rc != KW_OK) return rc;
    return estep_labels(N, x_dev, K, D, means_dev, prec_chol_dev, aux_dev, precision, w,
                        labels_dev, st);
}

extern "C" int kw_gmm_mstep_accumulate(int64_t N, const double* x_dev, int K, int D,
                                       const double* resp_dev, const double* centres_dev,
                                       double* stats_dev, int precision, int resp_form,
                                       void* workspace_dev, size_t workspace_bytes,
                                       void* stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    KW_REQUIRE(N > 0 && K > 0 && D > 0, "kw_gmm_mstep_accumulate: N, K, D must be positive");
    KW_REQUIRE(precision == 0 || precision == 1, "GMM precision must be 0 (fp64) or 1 (tensor)");
    KW_REQUIRE(resp_form == 0 || resp_form == 1, "resp_form must be 0 or 1");
    if (resp_form == 1 && precision == 0) {
        set_error("the FP64 M-step takes responsibilities: call kw_gmm_normalize_resp first");
        return KW_ERR_UNSUPPORTED;
    }
    if (D + 1 > 1024) {
        set_error("dim %d too large", D);
        return KW_ERR_UNSUPPORTED;
    }
    if (precision == 1 && D > GMM_MAX_DIM) return dim_unsupported("kw_gmm_mstep_accumulate", D);
    GmmWorkspace w;
    int rc = carve_fit(N, K, D, precision, workspace_dev, workspace_bytes, w);
    if (rc != KW_OK) return rc;
    if (precision == 1)
        return mstats_tc(N, K, D, resp_dev, centres_dev, stats_dev, w.tc, st, resp_form);
    return mstats_fp64(N, x_dev, K, D, resp_dev, centres_dev, w.partial, stats_dev, RESP_FLOOR, st);
}

extern "C" int kw_gmm_pack_frames(int64_t N, const double* x_dev, int K, int D, int precision,
                                  void* workspace_dev, size_t workspace_bytes, void* stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    KW_REQUIRE(N > 0 && K > 0 && D > 0, "kw_gmm_pack_frames: N, K, D must be positive");
    if (precision != 1) return KW_OK;
    if (D > GMM_MAX_DIM) return dim_unsupported("kw_gmm_pack_frames", D);
    GmmWorkspace w;
    int rc = carve_fit(N, K, D, precision, workspace_dev, workspace_bytes, w);
    if (rc != KW_OK) return rc;
    return pack_frames(N, x_dev, D, precision, w, st);
}

extern "C" int kw_gmm_mstep_finalize(int K, int D, double reg_covar, int weight_norm,
                                     const double* stats_dev, const double* centres_dev,
                                     double* weights_dev, double* means_dev,
                                     double* covariances_dev, double* prec_chol_dev,
                                     double* aux_dev, int32_t* info_dev, void* stream) {
    KW_REQUIRE(K > 0 && D > 0, "kw_gmm_mstep_finalize: K, D must be positive");
    return finalize_launch(K, D, reg_covar, weight_norm, 1, stats_dev, centres_dev, weights_dev,
                           means_dev, covariances_dev, prec_chol_dev, aux_dev, info_dev,
                           static_cast<cudaStream_t>(stream));
}

extern "C" int kw_gmm_precision_cholesky(int K, int D, const double* weights_dev,
                                         const double* means_dev, const double* covariances_dev,
                                         double* prec_chol_dev, double* aux_dev, int32_t* info_dev,
                                         void* stream) {
    KW_REQUIRE(K > 0 && D > 0, "kw_gmm_precision_cholesky: K, D must be positive");
    return finalize_launch(K, D, 0.0, 0, 0, nullptr, nullptr, const_cast<double*>(weights_dev),
                           const_cast<double*>(means_dev), const_cast<double*>(covariances_dev),
                           prec_chol_dev, aux_dev, info_dev, static_cast<cudaStream_t>(stream));
}

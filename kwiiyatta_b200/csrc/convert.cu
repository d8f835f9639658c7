// Conversion: hard posterior, conditional Gaussian, MLPG -- sm_100a, FP64.
//
// Replaces nnmnkwii.baseline.gmm.MLPG(gmm, windows, diff).transform(src) as called at
// kwiiyatta/converter/gmm.py:28-34 (restated in oracle/mlpg_ref.py):
//   m_t = argmax_k log N(x_t; mu_x, S_xx) + log w          (px.predict)
//   E_t = mu_y[m] + S_yx[m] S_xx[m]^-1 (x_t - mu_x[m])       = offset[m] + A[m] x_t
//   D_t = diag(S_yy[m]) - diag(S_yx[m]) / diag(S_xx[m]) * diag(S_xy[m])   (per mixture table)
//   y[:, d] = solve( W^T D^-1 W , W^T D^-1 E )  per static dim d, pentadiagonal SPD system,
//   windows = kwiiyatta DELTA_WINDOWS (kwiiyatta/converter/delta.py:8-12).
// Beyond the reference: global-variance (GV) statistics and GV-considered generation on the same
// normal equations (kw_gv_estimate, kw_convert_gv_batch; restated in oracle/gv_ref.py),
// maximum-likelihood conversion over all mixture sequences by EM (kw_convert_em_batch; restated
// in oracle/mlpg_em_ref.py), and the ML trajectory under the full conditional covariance
//   Sigma_m = S_yy - A_m S_xy  (Dh x Dh) in place of D_m, a block-pentadiagonal system with
// sd x sd blocks solved by a block Cholesky sweep per utterance (kw_convert_fullcov_batch;
// restated in oracle/mlpg_full_ref.py).  Its workspace keeps the block factors between the
// forward and the backward sweep: (3 sd^2 + sd) doubles per frame, 14 KB at sd = 24, where the
// diagonal path's band takes 768 B.
#include <vector>

#include "common.cuh"

namespace kw {

struct PreparedView {
    double* px_prec_chol;  // (K, Dh, Dh)
    double* px_aux;        // (K, Dh + 2)
    double* at;            // (K, Dh, Dh)  A^T: at[c][r] = A[r][c]
    double* offset;        // (K, Dh)
    double* var;           // (K, Dh)
    double* scratch;       // (K, Dh, Dh)  S_xx, then S_yx P
    double* src_means;     // (K, Dh)
    double* tgt_means;     // (K, Dh)
    size_t len;
};

static PreparedView view_prepared(double* base, int K, int Dh) {
    PreparedView v;
    size_t o = 0;
    const size_t kdd = (size_t)K * Dh * Dh, kd = (size_t)K * Dh;
    v.px_prec_chol = base + o; o += kdd;
    v.px_aux = base + o;       o += (size_t)K * (Dh + 2);
    v.at = base + o;           o += kdd;
    v.offset = base + o;       o += kd;
    v.var = base + o;          o += kd;
    v.scratch = base + o;      o += kdd;
    v.src_means = base + o;    o += kd;
    v.tgt_means = base + o;    o += kd;
    v.len = o;
    return v;
}

// Slice the joint model (MLPGBase.__init__), with the diff rewrite when asked.
__global__ void convert_slice_kernel(int K, int Dh, int diff, const double* __restrict__ means,
                                     const double* __restrict__ cov, PreparedView v) {
    const int k = blockIdx.x;
    const int D = 2 * Dh;
    const double* C = cov + (size_t)k * D * D;
    const double* mu = means + (size_t)k * D;
    for (int e = threadIdx.x; e < Dh * Dh; e += blockDim.x) {
        const int r = e / Dh, c = e - r * Dh;
        v.scratch[(size_t)k * Dh * Dh + e] = C[(size_t)r * D + c];  // S_xx
    }
    for (int d = threadIdx.x; d < Dh; d += blockDim.x) {
        const double cxx = C[(size_t)d * D + d];
        double cxy = C[(size_t)d * D + Dh + d];
        double cyx = C[(size_t)(Dh + d) * D + d];
        double cyy = C[(size_t)(Dh + d) * D + Dh + d];
        double ty = mu[Dh + d];
        if (diff) {
            ty = ty - mu[d];
            cyy = cxx + cyy - cxy - cyx;
            cxy = cxy - cxx;
            cyx = cxy;
        }
        v.src_means[(size_t)k * Dh + d] = mu[d];
        v.tgt_means[(size_t)k * Dh + d] = ty;
        v.var[(size_t)k * Dh + d] = cyy - cyx / cxx * cxy;
    }
}

// A = S_yx P P^T (P = px_prec_chol, upper), offset = mu_y - A mu_x.  One CTA per mixture.
__global__ void convert_regress_kernel(int K, int Dh, int diff, const double* __restrict__ cov,
                                       PreparedView v) {
    extern __shared__ double t1[];  // Dh * Dh : S_yx P
    const int k = blockIdx.x;
    const int D = 2 * Dh;
    const double* C = cov + (size_t)k * D * D;
    const double* P = v.px_prec_chol + (size_t)k * Dh * Dh;
    auto syx = [&](int r, int c) -> double {
        if (!diff) return C[(size_t)(Dh + r) * D + c];
        return C[(size_t)c * D + Dh + r] - C[(size_t)c * D + r];  // (S_xy - S_xx)^T
    };
    for (int e = threadIdx.x; e < Dh * Dh; e += blockDim.x) {
        const int r = e / Dh, c = e - r * Dh;
        double s = 0.0;
        for (int q = 0; q <= c; ++q) s = fma(syx(r, q), P[(size_t)q * Dh + c], s);
        t1[e] = s;
    }
    __syncthreads();
    double* at = v.at + (size_t)k * Dh * Dh;
    for (int e = threadIdx.x; e < Dh * Dh; e += blockDim.x) {
        const int r = e / Dh, c = e - r * Dh;
        double s = 0.0;
        for (int q = c; q < Dh; ++q) s = fma(t1[r * Dh + q], P[(size_t)c * Dh + q], s);
        at[(size_t)c * Dh + r] = s;
    }
    __syncthreads();
    const double* mx = v.src_means + (size_t)k * Dh;
    for (int r = threadIdx.x; r < Dh; r += blockDim.x) {
        double s = 0.0;
        for (int c = 0; c < Dh; ++c) s = fma(at[(size_t)c * Dh + r], mx[c], s);
        v.offset[(size_t)k * Dh + r] = v.tgt_means[(size_t)k * Dh + r] - s;
    }
}

// Conditional means E[t] = offset[m_t] + A[m_t] x[t], grouped by mixture: a counting sort of the
// frames by hard label (histogram, scan, scatter), then one CTA per (mixture, 64 frames of it)
// with A^T of that mixture and the frames staged in shared memory.
constexpr int CM_FT = 64;

__global__ void convert_hist_kernel(long long N, int K, const int32_t* __restrict__ mix,
                                    int* __restrict__ counts) {
    extern __shared__ int h[];
    for (int i = threadIdx.x; i < K; i += blockDim.x) h[i] = 0;
    __syncthreads();
    for (long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x; n < N;
         n += (long long)gridDim.x * blockDim.x)
        atomicAdd(&h[mix[n]], 1);
    __syncthreads();
    for (int i = threadIdx.x; i < K; i += blockDim.x)
        if (h[i] != 0) atomicAdd(&counts[i], h[i]);
}

// offsets[m] = first slot of mixture m in the sorted order; blockstart[m] = first CTA of it.
__global__ void convert_scan_kernel(int K, const int* __restrict__ counts, int* __restrict__ offsets,
                                    int* __restrict__ blockstart, int* __restrict__ cursor) {
    if (threadIdx.x == 0) {
        int o = 0, b = 0;
        for (int m = 0; m < K; ++m) {
            offsets[m] = o;
            blockstart[m] = b;
            cursor[m] = 0;
            o += counts[m];
            b += (counts[m] + CM_FT - 1) / CM_FT;
        }
        offsets[K] = o;
        blockstart[K] = b;
    }
}

__global__ void convert_scatter_kernel(long long N, const int32_t* __restrict__ mix,
                                       const int* __restrict__ offsets, int* __restrict__ cursor,
                                       int* __restrict__ order) {
    const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const int m = mix[n];
    order[offsets[m] + atomicAdd(&cursor[m], 1)] = (int)n;
}

__global__ void __launch_bounds__(256)
convert_condmean_kernel(int K, int Dh, const double* __restrict__ src,
                        const int* __restrict__ offsets, const int* __restrict__ blockstart,
                        const int* __restrict__ order, PreparedView v, double* __restrict__ E) {
    extern __shared__ double sm[];
    const int XS = Dh + 1;
    double* as = sm;                    // Dh * Dh : A^T[c][r]
    double* xs = as + Dh * Dh;          // CM_FT * XS
    __shared__ int idx[CM_FT];
    if ((int)blockIdx.x >= blockstart[K]) return;
    int lo = 0, hi = K;                 // mixture with blockstart[m] <= blockIdx.x < blockstart[m+1]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (blockstart[mid] <= (int)blockIdx.x) lo = mid; else hi = mid;
    }
    const int m = lo;
    const int first = offsets[m] + ((int)blockIdx.x - blockstart[m]) * CM_FT;
    const int count = min(CM_FT, offsets[m + 1] - first);
    const int tid = threadIdx.x;
    if (tid < CM_FT) idx[tid] = tid < count ? order[first + tid] : -1;
    const double* at = v.at + (size_t)m * Dh * Dh;
    for (int e = tid; e < Dh * Dh; e += 256) as[e] = at[e];
    __syncthreads();
    for (int e = tid; e < CM_FT * Dh; e += 256) {
        const int f = e / Dh, c = e - f * Dh;
        xs[f * XS + c] = idx[f] >= 0 ? src[(size_t)idx[f] * Dh + c] : 0.0;
    }
    __syncthreads();
    const int ty = tid >> 4, tx = tid & 15;
    double acc[4][5];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int q = 0; q < 5; ++q) acc[a][q] = 0.0;
    for (int c = 0; c < Dh; ++c) {
        double a[5], x[4];
#pragma unroll
        for (int q = 0; q < 5; ++q) a[q] = (tx + 16 * q < Dh) ? as[c * Dh + tx + 16 * q] : 0.0;
#pragma unroll
        for (int f = 0; f < 4; ++f) x[f] = xs[(ty * 4 + f) * XS + c];
#pragma unroll
        for (int f = 0; f < 4; ++f)
#pragma unroll
            for (int q = 0; q < 5; ++q) acc[f][q] = fma(a[q], x[f], acc[f][q]);
    }
    const double* off = v.offset + (size_t)m * Dh;
#pragma unroll
    for (int f = 0; f < 4; ++f) {
        const int n = idx[ty * 4 + f];
        if (n < 0) continue;
#pragma unroll
        for (int q = 0; q < 5; ++q) {
            const int r = tx + 16 * q;
            if (r < Dh) E[(size_t)n * Dh + r] = off[r] + acc[f][q];
        }
    }
}

// Soft-posterior mapping (nnmnkwii MLPGBase.transform, the mlpg=False branch of
// kwiiyatta/converter/gmm.py:30-31):  y_t = sum_m p(m | x_t) (offset[m] + A[m] x_t).
// CTA = 32 frames; thread r owns output dimension r for all 32 frames; mixtures whose posterior is
// not above SOFT_FLOOR for any frame of the tile are skipped.
// PREC (the M-step of EM conversion): every term is also weighted by 1 / var[m][r] and terms with
// p(m | x_t) <= SOFT_FLOOR are dropped, so out = q_t = sum_m p D_m^-1 E_{m,t} and prec_out =
// P_t = sum_m p D_m^-1 (both (N, Dh)).
constexpr int SOFT_FT = 32;
constexpr double SOFT_FLOOR = 1e-14;
template <bool PREC>
__global__ void __launch_bounds__(96)
convert_soft_kernel(long long N, long long Npad, int K, int Dh, const double* __restrict__ src,
                    const double* __restrict__ respT, PreparedView v, double* __restrict__ out,
                    double* __restrict__ prec_out) {
    extern __shared__ double xs[];          // SOFT_FT * Dh frames, then SOFT_FT responsibilities
    double* rs = xs + SOFT_FT * Dh;
    __shared__ int any_active;
    const long long n0 = (long long)blockIdx.x * SOFT_FT;
    for (int e = threadIdx.x; e < SOFT_FT * Dh; e += blockDim.x) {
        const long long n = n0 + e / Dh;
        xs[e] = (n < N) ? src[n * Dh + (e % Dh)] : 0.0;
    }
    const int r = threadIdx.x;
    double acc[SOFT_FT], pacc[PREC ? SOFT_FT : 1];
#pragma unroll
    for (int f = 0; f < SOFT_FT; ++f) acc[f] = 0.0;
    if (PREC) {
#pragma unroll
        for (int f = 0; f < SOFT_FT; ++f) pacc[f] = 0.0;
    }
    for (int m = 0; m < K; ++m) {
        __syncthreads();
        if (threadIdx.x == 0) any_active = 0;
        __syncthreads();
        if (threadIdx.x < SOFT_FT) {
            const long long n = n0 + threadIdx.x;
            const double p = (n < N) ? respT[(size_t)m * Npad + n] : 0.0;
            rs[threadIdx.x] = (PREC && !(p > SOFT_FLOOR)) ? 0.0 : p;
            if (p > SOFT_FLOOR) any_active = 1;
        }
        __syncthreads();
        if (!any_active || r >= Dh) continue;
        const double* at = v.at + (size_t)m * Dh * Dh;
        const double off = v.offset[(size_t)m * Dh + r];
        double e[SOFT_FT];
#pragma unroll
        for (int f = 0; f < SOFT_FT; ++f) e[f] = off;
        for (int c = 0; c < Dh; ++c) {
            const double a = at[(size_t)c * Dh + r];
#pragma unroll
            for (int f = 0; f < SOFT_FT; ++f) e[f] = fma(a, xs[f * Dh + c], e[f]);
        }
        if (PREC) {
            const double iv = 1.0 / v.var[(size_t)m * Dh + r];
#pragma unroll
            for (int f = 0; f < SOFT_FT; ++f) {
                const double g = rs[f] * iv;
                pacc[f] += g;
                acc[f] = fma(g, e[f], acc[f]);
            }
        } else {
#pragma unroll
            for (int f = 0; f < SOFT_FT; ++f) acc[f] = fma(rs[f], e[f], acc[f]);
        }
    }
    if (r < Dh) {
#pragma unroll
        for (int f = 0; f < SOFT_FT; ++f)
            if (n0 + f < N) {
                out[(n0 + f) * Dh + r] = acc[f];
                if (PREC) prec_out[(n0 + f) * Dh + r] = pacc[f];
            }
    }
}

// MLPG in two kernels.
//  1. convert_band_kernel, one thread per (frame, static dim): the pentadiagonal normal
//     equations W^T P W y = W^T P mu of that dimension, row by row: a_i = P[i][i],
//     b_i = P[i][i+1], c_i = P[i][i+2] and the right-hand side.  Fully parallel; this is where
//     the per-frame gathers (mixture -> variance) and the divisions happen.  FRAME_PREC (the
//     M-step of EM conversion) reads the per-frame precision P_t from `var` and the
//     precision-weighted mean P_t mu_t from `E`, both (total, Dh); `mix` is unused.
//  2. convert_mlpg_kernel, one thread per (utterance, static dim): banded Cholesky
//     (bandwidth 2) and the two substitutions, in place over the four arrays, reading four
//     steps ahead of the recurrence.  The chain per frame is two fused multiply-adds and one
//     reciprocal square root: with r_i = 1 / L[i][i], e_i = L[i][i-1], f_i = L[i][i-2]
//        f_i = c_{i-2} r_{i-2};  e_i = (b_{i-1} - f_i e_{i-1}) r_{i-1};
//        r_i = rsqrt(a_i - f_i^2 - e_i^2);  z_i = (rhs_i - e_i z_{i-1} - f_i z_{i-2}) r_i
//     and back:  y_i = (z_i - e_{i+1} y_{i+1} - f_{i+2} y_{i+2}) r_i  with f_{i+2} = c_i r_i.
struct Windows {
    double c[3][3];  // c[w][o+1]: coefficient of window w at offset o in {-1, 0, 1}
};

// flags[n]: bit 0 = first frame of its utterance, bit 1 = last frame
__global__ void convert_flags_kernel(int n_utts, const int64_t* __restrict__ off,
                                     unsigned char* __restrict__ flags) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= n_utts) return;
    const long long t0 = off[u], t1 = off[u + 1];
    if (t1 <= t0) return;
    if (t1 - t0 == 1) {
        flags[t0] = 3;
    } else {
        flags[t0] = 1;
        flags[t1 - 1] = 2;
    }
}

template <bool FRAME_PREC>
__global__ void __launch_bounds__(256)
convert_band_kernel(long long total, int sd, int Dh, const double* __restrict__ E,
                    const int32_t* __restrict__ mix, const double* __restrict__ var,
                    const unsigned char* __restrict__ flags, Windows win,
                    double* __restrict__ band) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= total * sd) return;
    const long long n = gid / sd;
    const int d = (int)(gid - n * sd);
    const unsigned fl = flags[n];
    // p[w], bs[w] at frames n-1 (m), n (c), n+1 (x)
    double pm[3] = {0, 0, 0}, bm[3] = {0, 0, 0}, pc[3], bc[3], px[3] = {0, 0, 0}, bx[3] = {0, 0, 0};
    auto load = [&](long long t, double* p, double* b) {
        if (FRAME_PREC) {
#pragma unroll
            for (int w = 0; w < 3; ++w) {
                p[w] = var[t * Dh + w * sd + d];
                b[w] = E[t * Dh + w * sd + d];
            }
            return;
        }
        const int m = mix[t];
#pragma unroll
        for (int w = 0; w < 3; ++w) {
            const double prec = 1.0 / var[(size_t)m * Dh + w * sd + d];
            p[w] = prec;
            b[w] = prec * E[t * Dh + w * sd + d];
        }
    };
    load(n, pc, bc);
    if (!(fl & 1u)) load(n - 1, pm, bm);
    if (!(fl & 2u)) load(n + 1, px, bx);
    double a_i = 0.0, b_i = 0.0, c_i = 0.0, rhs = 0.0;
#pragma unroll
    for (int w = 0; w < 3; ++w) {
        const double cm = win.c[w][0], c0 = win.c[w][1], cp = win.c[w][2];
        a_i += cp * cp * pm[w] + c0 * c0 * pc[w] + cm * cm * px[w];
        rhs += cp * bm[w] + c0 * bc[w] + cm * bx[w];
        b_i += c0 * cp * pc[w] + cm * c0 * px[w];
        c_i += cm * cp * px[w];
    }
    const size_t plane = (size_t)total * sd;
    band[gid] = a_i;
    band[plane + gid] = b_i;
    band[2 * plane + gid] = c_i;
    band[3 * plane + gid] = rhs;
}

__global__ void __launch_bounds__(96)
convert_mlpg_kernel(int n_utts, const int64_t* __restrict__ off, int sd, double* __restrict__ ws,
                    long long total, double* __restrict__ out) {
    const int gid = blockIdx.x * blockDim.x + threadIdx.x;
    const int u = gid / sd, d = gid - u * sd;
    if (u >= n_utts) return;
    const long long t0 = off[u];
    const int T = (int)(off[u + 1] - t0);
    if (T <= 0) return;
    const size_t plane = (size_t)total * sd;
    double* pa = ws + (size_t)t0 * sd + d;     // a -> r
    double* pb = pa + plane;                   // b -> e
    double* pcc = pb + plane;                  // c (kept)
    double* pr = pcc + plane;                  // rhs -> z
    constexpr int PF = 4;
    double c_m2 = 0, c_m1 = 0, b_m1 = 0, r_m1 = 1, r_m2 = 1, e_m1 = 0, z_m1 = 0, z_m2 = 0;
    double na[PF], nb[PF], nc[PF], nr[PF];
    auto fetch = [&](int i0) {
#pragma unroll
        for (int q = 0; q < PF; ++q) {
            const int i = min(i0 + q, T - 1);
            const size_t o = (size_t)i * sd;
            na[q] = pa[o]; nb[q] = pb[o]; nc[q] = pcc[o]; nr[q] = pr[o];
        }
    };
    fetch(0);
    for (int i0 = 0; i0 < T; i0 += PF) {
        double ca[PF], cb[PF], cc[PF], cr[PF];
#pragma unroll
        for (int q = 0; q < PF; ++q) { ca[q] = na[q]; cb[q] = nb[q]; cc[q] = nc[q]; cr[q] = nr[q]; }
        if (i0 + PF < T) fetch(i0 + PF);
#pragma unroll
        for (int q = 0; q < PF; ++q) {
            if (i0 + q < T) {
                const double f = c_m2 * r_m2;
                const double e = (b_m1 - f * e_m1) * r_m1;
                const double r = rsqrt(ca[q] - f * f - e * e);
                const double z = (cr[q] - e * z_m1 - f * z_m2) * r;
                const size_t o = (size_t)(i0 + q) * sd;
                pa[o] = r; pb[o] = e; pr[o] = z;      // c stays: f_{i+2} = c_i r_i on the way back
                c_m2 = c_m1; c_m1 = cc[q]; b_m1 = cb[q];
                r_m2 = r_m1; r_m1 = r; e_m1 = e;
                z_m2 = z_m1; z_m1 = z;
            }
        }
    }
    // back substitution L^T y = z
    double* po = out + (size_t)t0 * sd + d;
    double y1 = 0, y2 = 0, e_n1 = 0;
    auto fetch_back = [&](int i0) {      // steps i0, i0-1, ...
#pragma unroll
        for (int q = 0; q < PF; ++q) {
            const int i = max(i0 - q, 0);
            const size_t o = (size_t)i * sd;
            na[q] = pa[o]; nb[q] = pb[o]; nc[q] = pcc[o]; nr[q] = pr[o];
        }
    };
    fetch_back(T - 1);
    for (int i0 = T - 1; i0 >= 0; i0 -= PF) {
        double ca[PF], cb[PF], cc[PF], cr[PF];
#pragma unroll
        for (int q = 0; q < PF; ++q) { ca[q] = na[q]; cb[q] = nb[q]; cc[q] = nc[q]; cr[q] = nr[q]; }
        if (i0 - PF >= 0) fetch_back(i0 - PF);
#pragma unroll
        for (int q = 0; q < PF; ++q) {
            if (i0 - q >= 0) {
                const double y = (cr[q] - e_n1 * y1 - (cc[q] * ca[q]) * y2) * ca[q];
                po[(size_t)(i0 - q) * sd] = y;
                y2 = y1; y1 = y;
                e_n1 = cb[q];
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// Global variance (Toda, Black & Tokuda, IEEE TASLP 15(8), 2007; restated in oracle/gv_ref.py).
//
// kw_gv_estimate, one warp per (utterance, column): v = (1/T) sum_t (x_t - mean)^2 by two passes
// (mean, then squared deviations), lane-strided partial sums and an xor-butterfly, so every sum
// has one fixed order.  gv_reduce_kernel, one thread per column: mu_v, sigma^2_v over the
// utterances with T >= 1 in utterance order, plus [sum v | sum v^2 | count] for an all-reduce.
// (warp_sum's xor-butterfly leaves the same bits on every lane, so every lane takes the same
// accept / reject branch below.)
constexpr double GV_VAR_FLOOR = 1e-12;  // sigma^2_v floor: p = 1 / sigma^2_v stays finite

__global__ void gv_utt_var_kernel(int n_utts, const int64_t* __restrict__ off, int ld, int col0,
                                  int ncols, const double* __restrict__ x,
                                  double* __restrict__ utt_var) {
    const int warp = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (warp >= n_utts * ncols) return;
    const int u = warp / ncols, c = warp - u * ncols;
    const long long t0 = off[u];
    const int T = (int)(off[u + 1] - t0);
    const double* p = x + (size_t)t0 * ld + col0 + c;
    double s = 0.0;
    for (int t = lane; t < T; t += 32) s += p[(size_t)t * ld];
    const double mean = T > 0 ? warp_sum(s) / T : 0.0;
    double q = 0.0;
    for (int t = lane; t < T; t += 32) {
        const double e = p[(size_t)t * ld] - mean;
        q += e * e;
    }
    q = warp_sum(q);
    if (lane == 0) utt_var[(size_t)u * ncols + c] = T > 0 ? q / T : 0.0;
}

__global__ void gv_reduce_kernel(int n_utts, const int64_t* __restrict__ off, int ncols,
                                 const double* __restrict__ utt_var, double* __restrict__ sums,
                                 double* __restrict__ mean, double* __restrict__ var) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncols) return;
    double s = 0.0, s2 = 0.0;
    int n = 0;
    for (int u = 0; u < n_utts; ++u) {
        if (off[u + 1] <= off[u]) continue;
        const double v = utt_var[(size_t)u * ncols + c];
        s += v;
        s2 += v * v;
        ++n;
    }
    const double mu = n > 0 ? s / n : 0.0;
    double q = 0.0;
    for (int u = 0; u < n_utts; ++u) {
        if (off[u + 1] <= off[u]) continue;
        const double e = utt_var[(size_t)u * ncols + c] - mu;
        q += e * e;
    }
    if (sums != nullptr) {
        sums[c] = s;
        sums[ncols + c] = s2;
        if (c == 0) sums[2 * ncols] = n;
    }
    mean[c] = mu;
    var[c] = fmax(n > 0 ? q / n : 0.0, GV_VAR_FLOOR);
}

// mu_v, sigma^2_v from [sum v | sum v^2 | count] summed over ranks.
__global__ void gv_from_sums_kernel(int ncols, const double* __restrict__ sums,
                                    double* __restrict__ mean, double* __restrict__ var) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncols) return;
    const double n = sums[2 * ncols];
    const double mu = n > 0 ? sums[c] / n : 0.0;
    mean[c] = mu;
    var[c] = fmax(n > 0 ? sums[ncols + c] / n - mu * mu : 0.0, GV_VAR_FLOOR);
}

// GV-considered generation, one warp per (utterance, static dim), on the normal equations the
// band kernel built (R y = r: a = R[t][t], b = R[t][t+1], c = R[t][t+2]; the planes hold values
// past the utterance's end for b and c, which are masked here) and the ML solution y0 in `out`:
//   F(y) = w_traj (-1/2 y^T R y + y^T r) - w_gv 1/2 p (v(y) - mu_v)^2,   p = 1 / sigma^2_v
//   y <- mean(y0) + sqrt(mu_v / v(y0)) (y0 - mean(y0))     (unless T < 2 or v(y0) = 0)
//   gv_iter times: g = w_traj (r - R y) - w_gv p (v - mu_v) (2/T) (y - ybar),
//     delta_t = w_traj R_tt + w_gv (2p/T^2) max(0, (T-1)(v - mu_v) + 2 (y_t - ybar)^2),
//     d = step g / delta;  accept y + d (step *= 1.2) iff F(y + d) >= F(y), else step *= 0.5.
// The test takes dF = F(y + d) - F(y) in closed form from d rather than as the difference of two
// rounded values of F:
//   dF = w_traj (d^T (r - R y) - 1/2 d^T R d) - w_gv 1/2 p dv (2 (v - mu_v) + dv),
//   dv = (2/T) sum (y_t - ybar) d_t + (1/T) sum (d_t - dbar)^2,
// and "dF >= 0" is read up to the rounding of the gradient it rests on:
//   dF >= -tol,  tol = GV_ROUND (w_traj sum |d_t| (|r_t| + (|R| |y|)_t)
//                                + w_gv p (v + mu_v) (2/T) sum |d_t| |y_t - ybar|).
// Where y is stationary to rounding (T = 1 from the start: y0 is the optimum) r - R y is noise
// of either sign or exactly zero, depending on the order of the operations; the tolerance makes
// every such step F-neutral and accepted, so two correct implementations count the same steps.  Diff mode: the problem in z = s + y (r' = r + R s, z0 = y0 + s), y = z - s.
// The arrays a, b, c, r, y and the step d live in shared memory when T <= GV_SMEM_FRAMES
// (stride 1), otherwise in the band workspace, `out` and a step plane (stride sd).
constexpr int GV_SMEM_FRAMES = 1024;  // 6 arrays x 1024 doubles = 48 KB per warp
constexpr double GV_ROUND = 8.0 * 2.220446049250313e-16;  // 8 ulp-units of the gradient terms

struct GvArgs {
    const int64_t* off;
    int n_utts, sd, gv_iter, smem_frames;
    const double* mu;
    const double* var;
    double w_traj, w_gv;
    const double* s;  // diff mode: static source, row stride s_ld; else nullptr
    int s_ld;
    double* band;     // [a | b | c | rhs], (total, sd) each
    double* step;     // (total, sd) step plane for the global-memory branch
    double* out;      // (total, sd): y0 in, y out
    long long total;
    double* f_out;    // (n_utts, sd) or nullptr
    int32_t* acc_out; // (n_utts, sd) or nullptr
};

template <int STRIDE>  // 1: shared memory; 0: global memory, stride sd
__device__ void gv_solve(const GvArgs& g, int u, int d, int T, double* A, double* B, double* C,
                         double* R, double* Y, double* D, int gs) {
    const int st = STRIDE == 1 ? 1 : gs;
    const int lane = threadIdx.x & 31;
    auto Ry = [&](const double* v, int t, double* mag = nullptr) {  // (R v)_t [, (|R| |v|)_t]
        double p0 = A[(size_t)t * st] * v[(size_t)t * st];
        double s = p0, m = fabs(p0);
        auto add = [&](double r, double x) { s = fma(r, x, s); m = fma(fabs(r), fabs(x), m); };
        if (t >= 1) add(B[(size_t)(t - 1) * st], v[(size_t)(t - 1) * st]);
        if (t >= 2) add(C[(size_t)(t - 2) * st], v[(size_t)(t - 2) * st]);
        if (t + 1 < T) add(B[(size_t)t * st], v[(size_t)(t + 1) * st]);
        if (t + 2 < T) add(C[(size_t)t * st], v[(size_t)(t + 2) * st]);
        if (mag != nullptr) *mag = m;
        return s;
    };
    const double mu = g.mu[d], p = 1.0 / g.var[d], wt = g.w_traj, wg = g.w_gv;
    const double invT = 1.0 / T;
    if (g.s != nullptr) {  // r' = r + R s, z0 = y0 + s; D holds s meanwhile
        const double* s = g.s + (size_t)g.off[u] * g.s_ld + d;
        for (int t = lane; t < T; t += 32) D[(size_t)t * st] = s[(size_t)t * g.s_ld];
        __syncwarp();
        for (int t = lane; t < T; t += 32) {
            R[(size_t)t * st] += Ry(D, t);
            Y[(size_t)t * st] += D[(size_t)t * st];
        }
        __syncwarp();
    }
    auto moments = [&](double& mean, double& v) {
        double s = 0.0;
        for (int t = lane; t < T; t += 32) s += Y[(size_t)t * st];
        mean = warp_sum(s) * invT;
        double q = 0.0;
        for (int t = lane; t < T; t += 32) {
            const double e = Y[(size_t)t * st] - mean;
            q = fma(e, e, q);
        }
        v = warp_sum(q) * invT;
    };
    double ybar, v;
    moments(ybar, v);
    if (T >= 2 && v > 0.0) {  // variance scaling: the postfilter and the start point
        const double k = sqrt(mu / v);
        for (int t = lane; t < T; t += 32) Y[(size_t)t * st] = ybar + k * (Y[(size_t)t * st] - ybar);
        __syncwarp();
        moments(ybar, v);
    }
    double step = 0.1;
    int accepted = 0;
    for (int it = 0; it < g.gv_iter; ++it) {
        const double gvc = wg * p * (v - mu);          // w_gv p (v - mu)
        double s_d = 0.0, s_dg = 0.0, s_yd = 0.0, s_et = 0.0, s_eg = 0.0;
        for (int t = lane; t < T; t += 32) {
            const double y = Y[(size_t)t * st], e = y - ybar;
            double mag;
            const double rt = R[(size_t)t * st];
            const double gt = wt * (rt - Ry(Y, t, &mag));
            const double grad = gt - gvc * (2.0 * invT) * e;
            const double curv = wt * A[(size_t)t * st] +
                                wg * (2.0 * p * invT * invT) * fmax(0.0, (T - 1) * (v - mu) + 2.0 * e * e);
            const double dt = step * grad / curv;
            D[(size_t)t * st] = dt;
            s_d += dt;
            s_dg = fma(dt, gt, s_dg);
            s_yd = fma(e, dt, s_yd);
            s_et = fma(fabs(dt), fabs(rt) + mag, s_et);
            s_eg = fma(fabs(dt), fabs(e), s_eg);
        }
        s_d = warp_sum(s_d);
        s_dg = warp_sum(s_dg);
        s_yd = warp_sum(s_yd);
        s_et = warp_sum(s_et);
        s_eg = warp_sum(s_eg);
        __syncwarp();
        const double dbar = s_d * invT;
        double s_dRd = 0.0, s_dd = 0.0;
        for (int t = lane; t < T; t += 32) {
            const double dt = D[(size_t)t * st], e = dt - dbar;
            s_dRd = fma(dt, Ry(D, t), s_dRd);
            s_dd = fma(e, e, s_dd);
        }
        s_dRd = warp_sum(s_dRd);
        s_dd = warp_sum(s_dd);
        const double dv = 2.0 * invT * s_yd + invT * s_dd;
        const double dF = s_dg - 0.5 * wt * s_dRd - 0.5 * wg * p * dv * (2.0 * (v - mu) + dv);
        const double tol = GV_ROUND * (wt * s_et + wg * p * (v + mu) * 2.0 * invT * s_eg);
        if (dF >= -tol) {
            for (int t = lane; t < T; t += 32) Y[(size_t)t * st] += D[(size_t)t * st];
            __syncwarp();
            moments(ybar, v);
            step *= 1.2;
            ++accepted;
        } else {
            step *= 0.5;
        }
        __syncwarp();
    }
    if (g.f_out != nullptr || g.acc_out != nullptr) {
        double s_f = 0.0;
        for (int t = lane; t < T; t += 32) {
            const double y = Y[(size_t)t * st];
            s_f = fma(y, R[(size_t)t * st] - 0.5 * Ry(Y, t), s_f);
        }
        s_f = warp_sum(s_f);
        if (lane == 0) {
            const double e = v - mu;
            if (g.f_out != nullptr) g.f_out[(size_t)u * g.sd + d] = wt * s_f - 0.5 * wg * p * e * e;
            if (g.acc_out != nullptr) g.acc_out[(size_t)u * g.sd + d] = accepted;
        }
    }
    __syncwarp();
    if (STRIDE == 1 || g.s != nullptr) {
        const double* s = g.s != nullptr ? g.s + (size_t)g.off[u] * g.s_ld + d : nullptr;
        double* o = g.out + (size_t)g.off[u] * g.sd + d;
        for (int t = lane; t < T; t += 32)
            o[(size_t)t * g.sd] = Y[(size_t)t * st] - (s != nullptr ? s[(size_t)t * g.s_ld] : 0.0);
    }
}

__global__ void __launch_bounds__(32)
convert_gv_kernel(GvArgs g) {
    extern __shared__ double gsm[];
    const int u = blockIdx.x / g.sd, d = blockIdx.x - u * g.sd;
    const long long t0 = g.off[u];
    const int T = (int)(g.off[u + 1] - t0);
    if (T <= 0) return;
    const int lane = threadIdx.x;
    const size_t plane = (size_t)g.total * g.sd;
    double* a = g.band + (size_t)t0 * g.sd + d;
    if (T <= g.smem_frames) {
        double* A = gsm;
        double* B = A + T;
        double* C = B + T;
        double* R = C + T;
        double* Y = R + T;
        double* D = Y + T;
        const double* y0 = g.out + (size_t)t0 * g.sd + d;
        for (int t = lane; t < T; t += 32) {
            const size_t o = (size_t)t * g.sd;
            A[t] = a[o]; B[t] = a[plane + o]; C[t] = a[2 * plane + o]; R[t] = a[3 * plane + o];
            Y[t] = y0[o];
        }
        __syncwarp();
        gv_solve<1>(g, u, d, T, A, B, C, R, Y, D, 1);
    } else {
        gv_solve<0>(g, u, d, T, a, a + plane, a + 2 * plane, a + 3 * plane,
                    g.out + (size_t)t0 * g.sd + d, g.step + (size_t)t0 * g.sd + d, g.sd);
    }
}

// ------------------------------------------------------------------------------------------
// Maximum-likelihood conversion over all mixture sequences (EM trajectory estimation; Toda,
// Black & Tokuda, IEEE TASLP 15(8), 2007; restated in oracle/mlpg_em_ref.py).  With the diagonal
// conditional variance the hard-sequence MLPG already uses, the model of the joint vector
// z_t = [x_t ; (W y)_t] under mixture m is ONE Gaussian of dimension 2 Dh:
//   mean [mu_x ; mu_y],  precision Cholesky (upper)  L~ = [[Lx, -A^T D^-1/2], [0, D^-1/2]],
//   log|L~| = log|Lx| - 1/2 sum_j log D_j,
// so the E-step is the GMM E-step at D = 2 Dh on z, and its per-frame log-normaliser summed over
// an utterance is the objective L(y) = sum_t log sum_m w_m N(x_t; mu_x, S_xx) N((W y)_t; E, D).
// M-step: P_t = sum_m g D_m^-1, q_t = sum_m g D_m^-1 E_{m,t} (g = gamma above SOFT_FLOOR), then
// (W^T P W) y = W^T q per static dimension, the MLPG system with per-frame precisions.

// The derived joint model (means, L~, aux = [mu~ L~ | log|L~| | log w]) from the prepared block.
// mu~ L~ = [mu_x Lx ; offset D^-1/2] (offset = mu_y - A mu_x).  One CTA per mixture.
__global__ void convert_em_model_kernel(int Dh, PreparedView v, double* __restrict__ means,
                                        double* __restrict__ pc, double* __restrict__ aux) {
    const int k = blockIdx.x;
    const int D = 2 * Dh;
    const double* lx = v.px_prec_chol + (size_t)k * Dh * Dh;
    const double* at = v.at + (size_t)k * Dh * Dh;
    const double* var = v.var + (size_t)k * Dh;
    double* L = pc + (size_t)k * D * D;
    for (int e = threadIdx.x; e < D * D; e += blockDim.x) {
        const int r = e / D, c = e - r * D;
        double x = 0.0;
        if (r < Dh && c < Dh) x = lx[r * Dh + c];
        else if (r < Dh) x = -at[r * Dh + c - Dh] / sqrt(var[c - Dh]);   // -A^T[r][j] / sqrt(D_j)
        else if (r == c) x = 1.0 / sqrt(var[r - Dh]);
        L[e] = x;
    }
    const double* pa = v.px_aux + (size_t)k * (Dh + 2);
    double* ak = aux + (size_t)k * (D + 2);
    for (int j = threadIdx.x; j < Dh; j += blockDim.x) {
        means[(size_t)k * D + j] = v.src_means[(size_t)k * Dh + j];
        means[(size_t)k * D + Dh + j] = v.tgt_means[(size_t)k * Dh + j];
        ak[j] = pa[j];
        ak[Dh + j] = v.offset[(size_t)k * Dh + j] / sqrt(var[j]);
    }
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int j = 0; j < Dh; ++j) s += log(var[j]);
        ak[D] = pa[Dh] - 0.5 * s;
        ak[D + 1] = pa[Dh + 1];
    }
}

// (W y)_t into columns [col0, col0 + 3 sd) of the row-major (total, ld) joint frames: window w at
// offsets -1, 0, +1, zero past the utterance's edges (flags), one thread per (frame, static dim).
__global__ void convert_em_frames_kernel(long long total, int sd, const double* __restrict__ y,
                                         const unsigned char* __restrict__ flags, Windows win,
                                         int ld, int col0, double* __restrict__ z) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= total * sd) return;
    const long long n = gid / sd;
    const int d = (int)(gid - n * sd);
    const unsigned fl = flags[n];
    const double yc = y[gid];
    const double ym = (fl & 1u) ? 0.0 : y[gid - sd];
    const double yp = (fl & 2u) ? 0.0 : y[gid + sd];
    double* o = z + n * ld + col0 + d;
#pragma unroll
    for (int w = 0; w < 3; ++w) o[w * sd] = win.c[w][0] * ym + win.c[w][1] * yc + win.c[w][2] * yp;
}

// out[u * stride + col] = sum of lse over the frames of utterance u: one warp per utterance,
// lane-strided partial sums and an xor-butterfly (one fixed order).
__global__ void convert_em_loglik_kernel(int n_utts, const int64_t* __restrict__ off,
                                         const double* __restrict__ lse, int stride, int col,
                                         double* __restrict__ out) {
    const int u = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (u >= n_utts) return;
    double s = 0.0;
    for (long long t = off[u] + lane; t < off[u + 1]; t += 32) s += lse[t];
    s = warp_sum(s);
    if (lane == 0) out[(size_t)u * stride + col] = s;
}

// ------------------------------------------------------------------------------------------
// Full conditional covariance (the ML trajectory of Toda, Black & Tokuda, IEEE TASLP 15(8), 2007;
// restated in oracle/mlpg_full_ref.py).  Per mixture Sigma_m = S_yy - A_m S_xy (Dh x Dh, after
// the diff rewrite), P_m = Sigma_m^-1 in 3 x 3 blocks P^(w,v) of sd x sd, and
//   G_m[a][b] = sum_{w,v} c[w][a+1] c[v][b+1] P^(w,v),   a, b in {-1, 0, 1}
// frame t adds G_{m_t}[a][b] to block (t+a, t+b) of R and sum_w c[w][a+1] g_t^(w) to block row
// t+a of r, g_t = P E_t = h_m + B_m x_t (B = P A, h = P offset); blocks outside [0, T) are
// dropped.  R y = r is block-pentadiagonal SPD with sd x sd blocks and couples the static
// dimensions, which the diagonal path (convert_band_kernel / convert_mlpg_kernel) solves apart.

// The fullcov block (kw_convert_fullcov_prepare), separate from the prepared block.
struct FullcovView {
    double* g;       // (K, FC_NG, sd, sd) G blocks, each column-major: [l * sd + k] = G[k][l]
    double* bt;      // (K, Dh, Dh) B^T, the layout of PreparedView::at
    double* h;       // (K, Dh)
    size_t len;
};

// The workspace of kw_convert_fullcov_prepare.
struct FullcovScratch {
    double* sigma;   // (K, Dh, Dh) Sigma
    double* pc;      // (K, Dh, Dh) precision Cholesky of Sigma (upper, P = pc pc^T)
    double* aux;     // (K, Dh + 2) by-product of the factorisation, unused
    double* ones;    // (K) unit weights for the factorisation
    size_t bytes;
};

static FullcovScratch carve_fullcov_scratch(int K, int Dh, void* base) {
    Carver c(base);
    FullcovScratch w;
    w.sigma = c.take<double>((size_t)K * Dh * Dh);
    w.pc = c.take<double>((size_t)K * Dh * Dh);
    w.aux = c.take<double>((size_t)K * (Dh + 2));
    w.ones = c.take<double>((size_t)K);
    w.bytes = align_up(c.used, 256);
    return w;
}

// The six distinct G blocks (G[b][a] = G[a][b]^T) in the order a frame's solve step reads them.
enum { FC_GMM, FC_G00, FC_GPP, FC_GP0, FC_G0M, FC_GPM, FC_NG };

static FullcovView view_fullcov(double* base, int K, int Dh) {
    FullcovView f;
    const int sd = Dh / 3;
    const size_t kdd = (size_t)K * Dh * Dh;
    size_t o = 0;
    f.g = base + o;     o += (size_t)K * FC_NG * sd * sd;
    f.bt = base + o;    o += kdd;
    f.h = base + o;     o += (size_t)K * Dh;
    f.len = o;
    return f;
}

// Sigma = S_yy - A S_xy, with the diff rewrite S_yy <- S_xx + S_yy - S_xy - S_yx,
// S_xy <- S_xy - S_xx.  One CTA per mixture.
__global__ void convert_fullcov_sigma_kernel(int Dh, int diff, const double* __restrict__ cov,
                                             PreparedView v, FullcovScratch w) {
    const int k = blockIdx.x;
    const int D = 2 * Dh;
    const double* C = cov + (size_t)k * D * D;
    const double* at = v.at + (size_t)k * Dh * Dh;
    for (int e = threadIdx.x; e < Dh * Dh; e += blockDim.x) {
        const int r = e / Dh, c = e - r * Dh;
        double s = C[(size_t)(Dh + r) * D + Dh + c];
        if (diff) s = C[(size_t)r * D + c] + s - C[(size_t)r * D + Dh + c] - C[(size_t)(Dh + r) * D + c];
        for (int q = 0; q < Dh; ++q) {
            double sxy = C[(size_t)q * D + Dh + c];
            if (diff) sxy -= C[(size_t)q * D + c];
            s = fma(-at[(size_t)q * Dh + r], sxy, s);
        }
        w.sigma[(size_t)k * Dh * Dh + e] = s;
    }
    if (threadIdx.x == 0) w.ones[k] = 1.0;
}

// P = pc pc^T, then the G blocks, B^T and h of one mixture.  One CTA per mixture, P in shared
// memory.
__global__ void convert_fullcov_tables_kernel(int Dh, PreparedView v, const double* __restrict__ pc,
                                              FullcovView f, Windows win) {
    extern __shared__ double P[];  // Dh * Dh
    const int k = blockIdx.x;
    const int sd = Dh / 3;
    const double* U = pc + (size_t)k * Dh * Dh;
    for (int e = threadIdx.x; e < Dh * Dh; e += blockDim.x) {
        const int r = e / Dh, c = e - r * Dh;
        double s = 0.0;
        for (int q = max(r, c); q < Dh; ++q) s = fma(U[(size_t)r * Dh + q], U[(size_t)c * Dh + q], s);
        P[e] = s;
    }
    __syncthreads();
    const int ss = sd * sd;
    for (int e = threadIdx.x; e < FC_NG * ss; e += blockDim.x) {
        const int blk = e / ss, rem = e - blk * ss;
        const int l = rem / sd, r = rem - l * sd;  // column-major: element G[r][l]
        const int a = blk == FC_GMM ? -1 : (blk == FC_G00 || blk == FC_G0M) ? 0 : 1;
        const int b = (blk == FC_GMM || blk == FC_G0M || blk == FC_GPM) ? -1 : blk == FC_GPP ? 1 : 0;
        double ca[3], cb[3];  // c[w][a + 1], c[w][b + 1] by selects: no dynamic index into win
#pragma unroll
        for (int w = 0; w < 3; ++w) {
            ca[w] = a < 0 ? win.c[w][0] : a == 0 ? win.c[w][1] : win.c[w][2];
            cb[w] = b < 0 ? win.c[w][0] : b == 0 ? win.c[w][1] : win.c[w][2];
        }
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < 3; ++w)
#pragma unroll
            for (int u = 0; u < 3; ++u)
                s = fma(ca[w] * cb[u], P[(w * sd + r) * Dh + u * sd + l], s);
        f.g[(size_t)k * FC_NG * ss + e] = s;
    }
    const double* at = v.at + (size_t)k * Dh * Dh;
    for (int e = threadIdx.x; e < Dh * Dh; e += blockDim.x) {
        const int c = e / Dh, r = e - c * Dh;  // B^T[c][r] = B[r][c] = sum_q P[r][q] A[q][c]
        double s = 0.0;
        for (int q = 0; q < Dh; ++q) s = fma(P[r * Dh + q], at[(size_t)c * Dh + q], s);
        f.bt[(size_t)k * Dh * Dh + e] = s;
    }
    const double* offset = v.offset + (size_t)k * Dh;
    for (int r = threadIdx.x; r < Dh; r += blockDim.x) {
        double s = 0.0;
        for (int q = 0; q < Dh; ++q) s = fma(P[r * Dh + q], offset[q], s);
        f.h[(size_t)k * Dh + r] = s;
    }
}

// The block solve, one warp per utterance; lane k owns row k of every sd x sd block.  Forward,
// block row i (right-looking block Cholesky):
//   A0 = R_ii + (updates of steps i-2, i-1),  A1 = R_{i+1,i} + (update of step i-1),  A2 = R_{i+2,i}
//   L_ii = chol(A0), L1 = A1 L_ii^-T, L2 = A2 L_ii^-T, z_i = L_ii^-1 (r_i + carried terms)
// as ONE column sweep over the 3 sd x sd panel [A0; A1; A2] and the right-hand side (lane k keeps
// its rows of A0, A1, A2 in registers; column j of L_ii is broadcast through shared memory), then
//   R~_{i+1,i+1} -= L1 L1^T,  R~_{i+2,i+2} = -L2 L2^T,  R~_{i+2,i+1} = -L2 L1^T
// (rows in registers / shared memory), and L_ii (diagonal stored as 1 / L_kk), L1, L2 and z_i go
// to the chain workspace, (3 sd^2 + sd) doubles per frame, column-major so the lanes store
// coalesced.  Back:  y_i = L_ii^-T (z_i - L1^T y_{i+1} - L2^T y_{i+2}).
// SDM: the largest static dimension the instantiation holds; EXACT: sd == SDM (no guards).
constexpr int FC_MAXSD = 26;  // dim_half <= 80, a multiple of 3

template <int SDM, bool EXACT>
__global__ void __launch_bounds__(32)
convert_fullcov_solve_kernel(const int64_t* __restrict__ off, int sd_arg,
                             const int32_t* __restrict__ mix, const double* __restrict__ g,
                             const double* __restrict__ gtab, Windows win,
                             double* __restrict__ chain, double* __restrict__ out) {
    constexpr int LD = SDM + 1;
    constexpr unsigned FULL = 0xffffffffu;
    __shared__ double Ls[SDM * LD];    // [l * LD + k]: L_ii[k][l] (back: the staged frame)
    __shared__ double L1s[SDM * LD];   // L1[k][l]
    __shared__ double L2s[SDM * LD];   // L2[k][l]
    __shared__ double accN[SDM * LD];  // lane k's row of the update of R_{i+1,i+1} (own row only)
    __shared__ double accO[SDM * LD];  // lane k's row of the update of R_{i+1,i}
    const int sd = EXACT ? SDM : sd_arg;
    const int u = blockIdx.x, k = threadIdx.x;
    const long long t0 = off[u];
    const int T = (int)(off[u + 1] - t0);
    if (T <= 0) return;
    const bool row = k < sd;
    const int Dh = 3 * sd;
    const size_t ss = (size_t)sd * sd, fs = 3 * ss + sd;
    double a0[SDM], a1[SDM], a2[SDM];
#pragma unroll
    for (int l = 0; l < SDM; ++l) {
        a0[l] = 0.0;
        if (row && l < sd) accN[l * LD + k] = accO[l * LD + k] = 0.0;
    }
    double rN = 0.0, rNN = 0.0;  // carried right-hand-side terms of rows i+1, i+2
    for (int i = 0; i < T; ++i) {
        const long long n = t0 + i;
        const bool hm = i >= 1, hp = i + 1 < T, hpp = i + 2 < T;
        double b = 0.0;
        if (row) {
            const double* G0 = gtab + (size_t)mix[n] * FC_NG * ss + k;
            const double* Gm = gtab + (size_t)(hm ? mix[n - 1] : 0) * FC_NG * ss + k;
            const double* Gp = gtab + (size_t)(hp ? mix[n + 1] : 0) * FC_NG * ss + k;
#pragma unroll
            for (int l = 0; l < SDM; ++l) {
                if (!EXACT && l >= sd) continue;
                const size_t o = (size_t)l * sd;
                double x = a0[l] + G0[FC_G00 * ss + o];
                if (hm) x += Gm[FC_GPP * ss + o];
                if (hp) x += Gp[FC_GMM * ss + o];
                a0[l] = x;
                a1[l] = hp ? accO[l * LD + k] + G0[FC_GP0 * ss + o] + Gp[FC_G0M * ss + o] : 0.0;
                a2[l] = hpp ? Gp[FC_GPM * ss + o] : 0.0;
            }
            const double* gc = g + (size_t)n * Dh + k;
            b = rN;
#pragma unroll
            for (int w = 0; w < 3; ++w) {
                b = fma(win.c[w][1], gc[w * sd], b);
                if (hm) b = fma(win.c[w][2], gc[w * sd - Dh], b);
                if (hp) b = fma(win.c[w][0], gc[w * sd + Dh], b);
            }
        } else {
#pragma unroll
            for (int l = 0; l < SDM; ++l) a0[l] = a1[l] = a2[l] = 0.0;
        }
        // column sweep: POTRF of A0, the two TRSMs and the forward substitution
        double inv_k = 0.0, z_k = 0.0, rN_next = rNN, rNN_next = 0.0;
#pragma unroll
        for (int j = 0; j < SDM; ++j) {
            if (!EXACT && j >= sd) continue;
            const double inv = rsqrt(__shfl_sync(FULL, a0[j], j));  // 1 / L_jj
            const double l0 = k >= j ? a0[j] * inv : 0.0;
            const double l1 = a1[j] * inv, l2 = a2[j] * inv;
            const double zj = __shfl_sync(FULL, b, j) * inv;
            if (k == j) { inv_k = inv; z_k = zj; }
            a0[j] = l0;
            a1[j] = l1;
            a2[j] = l2;
            if (k > j) b = fma(-l0, zj, b);
            rN_next = fma(-l1, zj, rN_next);
            rNN_next = fma(-l2, zj, rNN_next);
            if (row) Ls[j * LD + k] = l0;
            __syncwarp();
#pragma unroll
            for (int l = j + 1; l < SDM; ++l) {
                if (!EXACT && l >= sd) continue;
                const double L = Ls[j * LD + l];
                a0[l] = fma(-l0, L, a0[l]);
                a1[l] = fma(-l1, L, a1[l]);
                a2[l] = fma(-l2, L, a2[l]);
            }
        }
        rN = rN_next;
        rNN = rNN_next;
        if (row) {
            double* cf = chain + (size_t)n * fs + k;
#pragma unroll
            for (int l = 0; l < SDM; ++l) {
                if (!EXACT && l >= sd) continue;
                cf[(size_t)l * sd] = l == k ? inv_k : a0[l];
                cf[ss + (size_t)l * sd] = a1[l];
                cf[2 * ss + (size_t)l * sd] = a2[l];
                L1s[l * LD + k] = a1[l];
                L2s[l * LD + k] = a2[l];
            }
            cf[3 * ss] = z_k;
        }
        __syncwarp();
        // the SYRK / GEMM updates; a0 becomes the next step's update of its diagonal block
        if (row) {
#pragma unroll
            for (int j = 0; j < SDM; ++j) {
                if (!EXACT && j >= sd) continue;
                double d1 = 0.0, d2 = 0.0, d3 = 0.0;
#pragma unroll
                for (int l = 0; l < SDM; ++l) {
                    if (!EXACT && l >= sd) continue;
                    const double p = L1s[l * LD + j], q = L2s[l * LD + j];
                    d1 = fma(a1[l], p, d1);
                    d2 = fma(a2[l], q, d2);
                    d3 = fma(a2[l], p, d3);
                }
                a0[j] = accN[j * LD + k] - d1;
                accN[j * LD + k] = -d2;
                accO[j * LD + k] = -d3;
            }
        }
    }
    __syncwarp();
    double y1 = 0.0, y2 = 0.0;  // lane k: y_{i+1}[k], y_{i+2}[k]
    for (int i = T - 1; i >= 0; --i) {
        const double* cf = chain + (size_t)(t0 + i) * fs;
        for (int e = k; e < (int)ss; e += 32) {
            const int l = e / sd, r = e - l * sd;
            Ls[l * LD + r] = cf[e];
            L1s[l * LD + r] = cf[ss + e];
            L2s[l * LD + r] = cf[2 * ss + e];
        }
        __syncwarp();
        double b = row ? cf[3 * ss + k] : 0.0;
#pragma unroll
        for (int l = 0; l < SDM; ++l) {
            if (!EXACT && l >= sd) continue;
            const double p = __shfl_sync(FULL, y1, l), q = __shfl_sync(FULL, y2, l);
            if (row) b = fma(-L1s[k * LD + l], p, fma(-L2s[k * LD + l], q, b));  // L1[l][k], L2[l][k]
        }
        double y_k = 0.0;
#pragma unroll
        for (int j = SDM - 1; j >= 0; --j) {
            if (!EXACT && j >= sd) continue;
            const double yj = __shfl_sync(FULL, b, j) * Ls[j * LD + j];
            if (k == j) y_k = yj;
            if (k < j) b = fma(-Ls[k * LD + j], yj, b);  // L_ii[j][k]
        }
        if (row) out[(size_t)(t0 + i) * sd + k] = y_k;
        y2 = y1;
        y1 = y_k;
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------
// Low-delay conversion (fixed-lag MLPG; Muramatsu et al., Interspeech 2008; restated in
// oracle/mlpg_stream_ref.py) over many concurrent streams ("slots").  A stream delivers one static
// frame per call.  Delivering static j completes the source vector x_{j-1} (its deltas need
// static j), and with it the conditional mean and variance of frame j-1, so n = j frames are
// known.  The emitted frame is y^(n)[n-1-L], y^(n) the MLPG solution of frames [0, n).
// The system of [0, n) is the leading n x n block of the whole utterance's system except on row
// n-1, which lacks frame n's terms on its diagonal and right-hand side.  So rows 0 .. n-2 of the
// banded Cholesky factor are final and are carried forward one row per call with the recurrence
// of convert_mlpg_kernel; row n-1 is formed provisionally (it is final when the stream ends), and
// L + 1 steps of back substitution over a ring of the last factor rows give y^(n)[n-1-L].
// Band entries and factor steps use the expressions of convert_band_kernel and
// convert_mlpg_kernel, so with L >= T-1 a stream reproduces the offline conversion.

// The state of n_slots streams (kw_convert_stream_state_len doubles).  Per (slot, static dim):
// the last two statics, the precision terms p_w = 1 / D_w and b_w = p_w E_w of the last two
// completed frames, and a ring of L + 2 factor rows (r = 1 / L_ii, e = L_{i,i-1}, z, c = R_{i,i+2});
// frame / static / row i sits at i mod 2 (i mod (L + 2) in the ring).  Planes are (n_slots, sd).
struct StreamState {
    long long* count;  // (n_slots) statics delivered so far; 0 = empty slot
    double* statics;   // (2, n_slots, sd)
    double* terms;     // (2, 6, n_slots, sd): p_0, p_1, p_2, b_0, b_1, b_2
    double* ring;      // (L + 2, 4, n_slots, sd): r, e, z, c
    size_t len;        // in doubles
};

static StreamState view_stream_state(double* base, int n_slots, int sd, int delay) {
    StreamState s;
    const size_t plane = (size_t)n_slots * sd;
    size_t o = 0;
    s.count = reinterpret_cast<long long*>(base);  o += (size_t)n_slots;
    s.statics = base + o;                          o += 2 * plane;
    s.terms = base + o;                            o += 12 * plane;
    s.ring = base + o;                             o += ((size_t)delay + 2) * 4 * plane;
    s.len = o;
    return s;
}

// Source vectors: one warp per slot row i, lane d < sd.  x_{j-1} = [x~, delta, delta^2] of the
// statics j-2, j-1, j (zero outside [0, T); j = the static this call delivers, at the end the
// missing one), in kw_delta_features' order of operations; rows of slots with no complete frame
// get zeros.  Records j per row, stores static j and counts it (the end call empties the slot).
__global__ void convert_stream_source_kernel(int m, int sd, int end, const int* __restrict__ slots,
                                             const double* __restrict__ statics_in, StreamState s,
                                             int n_slots, double* __restrict__ x,
                                             long long* __restrict__ jrow) {
    const int i = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5);
    const int d = threadIdx.x & 31;
    if (i >= m) return;
    const int slot = slots[i];
    const long long j = s.count[slot];
    const size_t plane = (size_t)n_slots * sd;
    if (d < sd) {
        const size_t o = (size_t)slot * sd + d;
        const double xm = j >= 2 ? s.statics[((j - 2) & 1) * plane + o] : 0.0;
        const double xc = j >= 1 ? s.statics[((j - 1) & 1) * plane + o] : 0.0;
        const double xp = end ? 0.0 : statics_in[(size_t)i * sd + d];
        double* row = x + (size_t)i * 3 * sd;
        row[d] = xc;
        row[sd + d] = __dadd_rn(__dadd_rn(__dmul_rn(-0.5, xm), __dmul_rn(0.0, xc)), __dmul_rn(0.5, xp));
        row[2 * sd + d] = __dadd_rn(__dadd_rn(xm, __dmul_rn(-2.0, xc)), xp);
        if (!end) s.statics[(j & 1) * plane + o] = xp;   // replaces static j - 2, read above
    }
    __syncwarp();
    if (d == 0) {
        jrow[i] = j;
        s.count[slot] = end ? 0 : j + 1;
    }
}

// One row of the band from the precision terms of frames i-1 (m), i (c), i+1 (x): the expressions
// of convert_band_kernel.
__device__ __forceinline__ void stream_band_row(const double* pm, const double* bm, const double* pc,
                                                const double* bc, const double* px, const double* bx,
                                                const Windows& win, double& a, double& b, double& c,
                                                double& rhs) {
    a = 0.0; b = 0.0; c = 0.0; rhs = 0.0;
#pragma unroll
    for (int w = 0; w < 3; ++w) {
        const double cm = win.c[w][0], c0 = win.c[w][1], cp = win.c[w][2];
        a += cp * cp * pm[w] + c0 * c0 * pc[w] + cm * cm * px[w];
        rhs += cp * bm[w] + c0 * bc[w] + cm * bx[w];
        b += c0 * cp * pc[w] + cm * c0 * px[w];
        c += cm * cp * px[w];
    }
}

struct StreamStepArgs {
    int m, n_slots, sd, Dh, delay;
    const int* slots;
    const long long* jrow;
    const int32_t* mix;
    const double* E;
    const double* var;   // PreparedView::var
    StreamState s;
    Windows win;
    double* out;         // push: (m, sd); end: (m, delay + 1, sd)
    int64_t* index;      // push: emitted frame per row or -1; end: frames emitted per row
};

// One thread per (slot row, static dim).  Frame j-1 completes (n = j): row n-2 of the factor is
// finalised into the ring, row n-1 is formed from frames n-2 and n-1 alone, and the back
// substitution runs down to row max(0, n-1-L).  Push (END false): writes y^(n)[n-1-L] when that
// frame exists.  End (END true): row n-1 is final, and y^(n) of the last min(n, L+1) frames is
// written in order, zero rows after them.
template <bool END>
__global__ void __launch_bounds__(128) convert_stream_step_kernel(StreamStepArgs g) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (long long)g.m * g.sd) return;
    const int i = (int)(gid / g.sd), d = (int)(gid - (long long)i * g.sd);
    const int sd = g.sd, L = g.delay, R = L + 2;
    const long long j = g.jrow[i];
    const size_t plane = (size_t)g.n_slots * sd;
    const size_t o = (size_t)g.slots[i] * sd + d;
    double* outp = END ? g.out + (size_t)i * (L + 1) * sd + d : g.out + (size_t)i * sd + d;
    if (j == 0) {                     // nothing complete yet (push) / an empty slot (end)
        if (END) {
            for (int k = 0; k <= L; ++k) outp[(size_t)k * sd] = 0.0;
        } else {
            outp[0] = 0.0;
        }
        if (d == 0) g.index[i] = END ? 0 : -1;
        return;
    }
    // precision terms of frames j-3 (m), j-2 (c) and the new frame j-1 (x)
    double pm[3] = {0, 0, 0}, bm[3] = {0, 0, 0}, pc[3] = {0, 0, 0}, bc[3] = {0, 0, 0}, px[3], bx[3];
    const int mx = g.mix[i];
#pragma unroll
    for (int w = 0; w < 3; ++w) {
        const double prec = 1.0 / g.var[(size_t)mx * g.Dh + w * sd + d];
        px[w] = prec;
        bx[w] = prec * g.E[(size_t)i * g.Dh + w * sd + d];
    }
    double* t_c = g.s.terms + ((j - 2) & 1) * 6 * plane + o;
    double* t_m = g.s.terms + ((j - 3) & 1) * 6 * plane + o;   // = frame j-1's place
#pragma unroll
    for (int w = 0; w < 3; ++w) {
        if (j >= 2) { pc[w] = t_c[w * plane]; bc[w] = t_c[(3 + w) * plane]; }
        if (j >= 3) { pm[w] = t_m[w * plane]; bm[w] = t_m[(3 + w) * plane]; }
    }
    if (!END) {
#pragma unroll
        for (int w = 0; w < 3; ++w) { t_m[w * plane] = px[w]; t_m[(3 + w) * plane] = bx[w]; }
    }
    double* ring = g.s.ring + o;
    auto row_at = [&](long long r) -> double* { return ring + (size_t)(r % R) * 4 * plane; };
    // the recurrence's carries: rows i-2 (_m2) and i-1 (_m1) of the row i it steps to, with the
    // initial values of convert_mlpg_kernel before row 0
    double c_m2 = 0, c_m1 = 0, b_m1 = 0, r_m1 = 1, r_m2 = 1, e_m1 = 0, z_m1 = 0, z_m2 = 0;
    if (j >= 2) {                     // finalise row j-2: frames j-3, j-2, j-1 are all in
        if (j >= 4) {
            const double* p = row_at(j - 4);
            r_m1 = p[0]; z_m1 = p[2 * plane]; c_m1 = p[3 * plane];
        }
        if (j >= 3) {
            const double* p = row_at(j - 3);
            c_m2 = c_m1; r_m2 = r_m1; z_m2 = z_m1;
            r_m1 = p[0]; e_m1 = p[plane]; z_m1 = p[2 * plane]; c_m1 = p[3 * plane];
            const double zero[3] = {0, 0, 0};
            double a_, c_, rhs_;
            stream_band_row(zero, zero, pm, bm, pc, bc, g.win, a_, b_m1, c_, rhs_);  // b_{j-3}
        }
        double a, b, c, rhs;
        stream_band_row(pm, bm, pc, bc, px, bx, g.win, a, b, c, rhs);
        const double f = c_m2 * r_m2;
        const double e = (b_m1 - f * e_m1) * r_m1;
        const double r = rsqrt(a - f * f - e * e);
        const double z = (rhs - e * z_m1 - f * z_m2) * r;
        double* p = row_at(j - 2);
        p[0] = r; p[plane] = e; p[2 * plane] = z; p[3 * plane] = c;
        c_m2 = c_m1; c_m1 = c; b_m1 = b;
        r_m2 = r_m1; r_m1 = r; e_m1 = e;
        z_m2 = z_m1; z_m1 = z;
    }
    // row j-1 from frames j-2 and j-1 (frame j is not in yet; at the end there is none)
    const double zero[3] = {0, 0, 0};
    double a, b_, c, rhs;
    stream_band_row(pc, bc, px, bx, zero, zero, g.win, a, b_, c, rhs);
    const double f = c_m2 * r_m2;
    const double e = (b_m1 - f * e_m1) * r_m1;
    const double r = rsqrt(a - f * f - e * e);
    const double z = (rhs - e * z_m1 - f * z_m2) * r;
    // back substitution L^T y = z from row j-1 down to row lo
    const long long lo = j - 1 - L > 0 ? j - 1 - L : 0;
    double y = z * r;
    if (END) outp[(size_t)(j - 1 - lo) * sd] = y;
    double y1 = y, y2 = 0.0, e_n1 = e;
    for (long long k = j - 2; k >= lo; --k) {
        const double* p = row_at(k);
        const double rk = p[0], ek = p[plane], zk = p[2 * plane], ck = p[3 * plane];
        y = (zk - e_n1 * y1 - (ck * rk) * y2) * rk;
        if (END) outp[(size_t)(k - lo) * sd] = y;
        y2 = y1; y1 = y;
        e_n1 = ek;
    }
    if (END) {
        const int count = (int)(j - lo);
        for (int k = count; k <= L; ++k) outp[(size_t)k * sd] = 0.0;
        if (d == 0) g.index[i] = count;
    } else {
        const bool emit = j - 1 - L >= 0;
        outp[0] = emit ? y : 0.0;
        if (d == 0) g.index[i] = emit ? j - 1 - L : -1;
    }
}

// ------------------------------------------------------------------------------------------
// Host side of the hard-sequence conversions (kw_convert_batch, kw_convert_gv_batch,
// kw_convert_em_batch, kw_convert_fullcov_batch): one workspace layout, one argument check and
// the stages they share.

enum ConvertKind { CONVERT_PLAIN, CONVERT_GV, CONVERT_EM, CONVERT_FULLCOV, CONVERT_STREAM };

// The workspace of one conversion call, in this order: the hard-sequence buffers every kind uses
// (the band set and the utterance flags except for the full-covariance kind, whose block solve
// takes neither, and the stream kind, which keeps its band in the stream state), then the GV
// step plane, the EM buffers, the block-solve chain or the stream's source rows, then the GMM
// layer's region of the E-steps the call runs: the hard-sequence labels at dim_half, and for EM
// also the posteriors at 2 * dim_half.
struct ConvertWorkspace {
    int32_t* mix;          // (total) hard mixture sequence
    int* counts;           // K      (counting sort of the frames by mixture)
    int* offsets;          // K + 1
    int* blockstart;       // K + 1
    int* cursor;           // K
    int* order;            // total
    double* E;             // (total, Dh) conditional means
    double* band;          // [a | b | c | rhs], (total, sd) each
    unsigned char* flags;  // (total) utterance edges
    double* step;          // GV: (total, sd) step plane
    double* z;             // EM: (total, 2 Dh) joint frames [x | W y]
    double* resp;          // EM: (K, resp_pad(total))
    double* lse;           // EM: (total) per-frame log-normaliser
    double* q;             // EM: (total, Dh)
    double* prec;          // EM: (total, Dh)
    double* means;         // EM: (K, 2 Dh)
    double* pc;            // EM: (K, 2 Dh, 2 Dh)
    double* aux;           // EM: (K, 2 Dh + 2)
    double* chain;         // full covariance: (total, 3 sd^2 + sd) block-Cholesky factors and z
    double* x;             // stream: (total, Dh) source vectors, one per slot row
    int* slots;            // stream: (total) the slots of the rows
    long long* jrow;       // stream: (total) the static each row delivers
    GmmWorkspace gmm;      // the E-steps
    size_t bytes;
};

static ConvertWorkspace carve_convert(ConvertKind kind, long long total, int K, int Dh,
                                      int precision, void* base) {
    const int sd = Dh / 3;
    Carver c(base);
    ConvertWorkspace w = {};
    w.mix = c.take<int32_t>((size_t)total);
    w.counts = c.take<int>((size_t)K);
    w.offsets = c.take<int>((size_t)K + 1);
    w.blockstart = c.take<int>((size_t)K + 1);
    w.cursor = c.take<int>((size_t)K);
    w.order = c.take<int>((size_t)total);
    w.E = c.take<double>((size_t)total * Dh);
    if (kind != CONVERT_FULLCOV && kind != CONVERT_STREAM) {
        w.band = c.take<double>(4 * (size_t)total * sd);
        w.flags = c.take<unsigned char>((size_t)total);
    }
    if (kind == CONVERT_GV) w.step = c.take<double>((size_t)total * sd);
    if (kind == CONVERT_EM) {
        const size_t D = 2 * (size_t)Dh;
        w.z = c.take<double>((size_t)total * D);
        w.resp = c.take<double>((size_t)K * (size_t)resp_pad(total));
        w.lse = c.take<double>((size_t)total);
        w.q = c.take<double>((size_t)total * Dh);
        w.prec = c.take<double>((size_t)total * Dh);
        w.means = c.take<double>((size_t)K * D);
        w.pc = c.take<double>((size_t)K * D * D);
        w.aux = c.take<double>((size_t)K * (D + 2));
    }
    if (kind == CONVERT_FULLCOV) w.chain = c.take<double>((size_t)total * (3 * (size_t)sd * sd + sd));
    if (kind == CONVERT_STREAM) {
        w.x = c.take<double>((size_t)total * Dh);
        w.slots = c.take<int>((size_t)total);
        w.jrow = c.take<long long>((size_t)total);
    }
    w.gmm = kind == CONVERT_EM ? carve_gmm(c, total, K, 2 * Dh, precision, GmmUse::Posterior)
                               : carve_gmm(c, total, K, Dh, precision, GmmUse::Labels);
    w.bytes = align_up(c.used, 256);
    return w;
}

// The arguments every conversion kind shares (the caller has returned early on an empty batch).
// estep_dim: the largest dimension an E-step of the call runs at.
static int check_convert(const char* fn, int n_utts, long long total, int K, int Dh, int precision,
                         int estep_dim) {
    KW_REQUIRE(n_utts > 0 && total > 0 && K > 0, "%s: bad sizes", fn);
    KW_REQUIRE(Dh % 3 == 0, "%s: dim_half %d is not static+delta+delta2 (multiple of 3)", fn, Dh);
    KW_REQUIRE(precision == 0 || precision == 1, "%s: precision must be 0 or 1", fn);
    if (estep_dim > GMM_MAX_DIM) {
        set_error("%s: dim_half %d: the E-step at dimension %d > %d is not supported", fn, Dh,
                  estep_dim, GMM_MAX_DIM);
        return KW_ERR_UNSUPPORTED;
    }
    KW_REQUIRE(Dh <= 80, "%s: dim_half %d > 80 unsupported", fn, Dh);
    KW_REQUIRE(total < 2147483647LL, "%s: too many frames for one conversion batch", fn);
    return KW_OK;
}

static int workspace_too_small(const char* fn, size_t need, size_t got) {
    set_error("%s: workspace too small: need %zu bytes, got %zu", fn, need, got);
    return KW_ERR_WORKSPACE;
}

static const Windows kDeltaWindows = {{{0.0, 1.0, 0.0}, {-0.5, 0.0, 0.5}, {1.0, -2.0, 1.0}}};

// The hard mixture sequence (the E-step in label mode) into w.mix, then the conditional means of
// the frames under it into w.E: a counting sort of the frames by mixture (histogram, scan,
// scatter) and one pass per mixture.
static int hard_sequence(long long total, const double* src, int K, int Dh, int precision,
                         const PreparedView& v, const ConvertWorkspace& w, cudaStream_t st) {
    int rc = pack_frames(total, src, Dh, precision, w.gmm, st, /*mstep_parts=*/false);
    if (rc == KW_OK)
        rc = estep_labels(total, src, K, Dh, v.src_means, v.px_prec_chol, v.px_aux, precision,
                          w.gmm, w.mix, st);
    if (rc != KW_OK) return rc;
    KW_CUDA_CHECK(cudaMemsetAsync(w.counts, 0, sizeof(int) * K, st));
    convert_hist_kernel<<<296, 256, sizeof(int) * K, st>>>(total, K, w.mix, w.counts);
    KW_CUDA_CHECK(cudaGetLastError());
    convert_scan_kernel<<<1, 32, 0, st>>>(K, w.counts, w.offsets, w.blockstart, w.cursor);
    KW_CUDA_CHECK(cudaGetLastError());
    convert_scatter_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(
        total, w.mix, w.offsets, w.cursor, w.order);
    KW_CUDA_CHECK(cudaGetLastError());
    const size_t smem = sizeof(double) * ((size_t)Dh * Dh + (size_t)CM_FT * (Dh + 1));
    KW_CUDA_CHECK(cudaFuncSetAttribute(convert_condmean_kernel,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const long long max_blocks = (total + CM_FT - 1) / CM_FT + K;
    convert_condmean_kernel<<<(unsigned)max_blocks, 256, smem, st>>>(
        K, Dh, src, w.offsets, w.blockstart, w.order, v, w.E);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

static int utterance_flags(int n_utts, const int64_t* off, long long total,
                           const ConvertWorkspace& w, cudaStream_t st) {
    KW_CUDA_CHECK(cudaMemsetAsync(w.flags, 0, (size_t)total, st));
    convert_flags_kernel<<<(n_utts + 127) / 128, 128, 0, st>>>(n_utts, off, w.flags);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

// The MLPG normal equations into w.band: from the conditional means w.E under the mixture
// sequence w.mix (FRAME_PREC false), or from the EM M-step's per-frame w.q and w.prec (true).
template <bool FRAME_PREC>
static int build_band(long long total, int Dh, const PreparedView& v, const ConvertWorkspace& w,
                      cudaStream_t st) {
    const int sd = Dh / 3;
    const long long cells = total * sd;
    convert_band_kernel<FRAME_PREC><<<(unsigned)((cells + 255) / 256), 256, 0, st>>>(
        total, sd, Dh, FRAME_PREC ? w.q : w.E, FRAME_PREC ? nullptr : w.mix,
        FRAME_PREC ? w.prec : v.var, w.flags, kDeltaWindows, w.band);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

// Solves the equations in w.band (factoring them in place) into out.
static int solve_mlpg(int n_utts, const int64_t* off, long long total, int Dh,
                      const ConvertWorkspace& w, double* out, cudaStream_t st) {
    const int sd = Dh / 3;
    const long long threads = (long long)n_utts * sd;
    convert_mlpg_kernel<<<(unsigned)((threads + 95) / 96), 96, 0, st>>>(n_utts, off, sd, w.band,
                                                                        total, out);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

// The block solve of the full-covariance system from the right-hand sides g_t in w.E under the
// mixture sequence w.mix, into out.
static int solve_fullcov(int n_utts, const int64_t* off, int Dh, const FullcovView& f,
                         const ConvertWorkspace& w, double* out, cudaStream_t st) {
    const int sd = Dh / 3;
    if (sd == 24)
        convert_fullcov_solve_kernel<24, true><<<n_utts, 32, 0, st>>>(
            off, sd, w.mix, w.E, f.g, kDeltaWindows, w.chain, out);
    else
        convert_fullcov_solve_kernel<FC_MAXSD, false><<<n_utts, 32, 0, st>>>(
            off, sd, w.mix, w.E, f.g, kDeltaWindows, w.chain, out);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

}  // namespace kw

using namespace kw;

extern "C" size_t kw_convert_prepared_len(int K, int Dh) {
    return view_prepared(nullptr, K, Dh).len;
}

extern "C" int kw_convert_prepare(int K, int Dh, int diff, const double* weights_dev,
                                  const double* means_dev, const double* covariances_dev,
                                  double* prepared_dev, int32_t* info_dev, void* stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    KW_REQUIRE(K > 0 && Dh > 0, "kw_convert_prepare: K, dim_half must be positive");
    PreparedView v = view_prepared(prepared_dev, K, Dh);
    convert_slice_kernel<<<K, 128, 0, st>>>(K, Dh, diff, means_dev, covariances_dev, v);
    KW_CUDA_CHECK(cudaGetLastError());
    int rc = finalize_launch(K, Dh, 0.0, 0, 0, nullptr, nullptr,
                             const_cast<double*>(weights_dev), v.src_means, v.scratch,
                             v.px_prec_chol, v.px_aux, info_dev, st);
    if (rc != KW_OK) return rc;
    const size_t smem = sizeof(double) * (size_t)Dh * Dh;
    KW_CUDA_CHECK(cudaFuncSetAttribute(convert_regress_kernel,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    convert_regress_kernel<<<K, 256, smem, st>>>(K, Dh, diff, covariances_dev, v);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

extern "C" size_t kw_convert_soft_workspace_bytes(int64_t total_frames, int K, int Dh) {
    Carver c(nullptr);
    c.take<double>((size_t)K * (size_t)resp_pad(total_frames));
    carve_gmm(c, total_frames, K, Dh, 0, GmmUse::Posterior);
    return align_up(c.used, 256);
}

extern "C" int kw_convert_soft_batch(int64_t total, const double* src_dev, int K, int Dh,
                                     const double* prepared_dev, double* out_dev,
                                     void* workspace_dev, size_t workspace_bytes, void* stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (total == 0) return KW_OK;
    KW_REQUIRE(total > 0 && K > 0 && Dh > 0, "kw_convert_soft_batch: bad sizes");
    KW_REQUIRE(Dh <= 96, "dim_half %d > 96 unsupported", Dh);
    if (kw_convert_soft_workspace_bytes(total, K, Dh) > workspace_bytes) {
        set_error("soft conversion workspace too small");
        return KW_ERR_WORKSPACE;
    }
    Carver c(workspace_dev);
    Posterior post;
    post.resp = c.take<double>((size_t)K * (size_t)resp_pad(total));
    const GmmWorkspace gmm = carve_gmm(c, total, K, Dh, 0, GmmUse::Posterior);
    PreparedView v = view_prepared(const_cast<double*>(prepared_dev), K, Dh);
    int rc = estep_posterior(total, src_dev, K, Dh, nullptr, v.px_prec_chol, v.px_aux, 0, gmm,
                             post, st);
    if (rc != KW_OK) return rc;
    const size_t smem = sizeof(double) * ((size_t)SOFT_FT * Dh + SOFT_FT);
    convert_soft_kernel<false><<<(unsigned)((total + SOFT_FT - 1) / SOFT_FT), 96, smem, st>>>(
        total, resp_pad(total), K, Dh, src_dev, post.resp, v, out_dev, nullptr);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

extern "C" size_t kw_convert_workspace_bytes(int64_t total_frames, int K, int Dh, int precision) {
    return carve_convert(CONVERT_PLAIN, total_frames, K, Dh, precision, nullptr).bytes;
}

extern "C" int kw_convert_batch(int n_utts, const int64_t* off_dev, int64_t total, int max_frames,
                                const double* src_dev, int K, int Dh, const double* prepared_dev,
                                double* out_dev, int32_t* mix_dev, int precision,
                                void* workspace_dev, size_t workspace_bytes, void* stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    (void)max_frames;
    if (n_utts == 0 || total == 0) return KW_OK;
    int rc = check_convert("kw_convert_batch", n_utts, total, K, Dh, precision, Dh);
    if (rc != KW_OK) return rc;
    const ConvertWorkspace w =
        carve_convert(CONVERT_PLAIN, total, K, Dh, precision, workspace_dev);
    if (w.bytes > workspace_bytes)
        return workspace_too_small("kw_convert_batch", w.bytes, workspace_bytes);
    const PreparedView v = view_prepared(const_cast<double*>(prepared_dev), K, Dh);
    rc = hard_sequence(total, src_dev, K, Dh, precision, v, w, st);
    if (rc == KW_OK) rc = utterance_flags(n_utts, off_dev, total, w, st);
    if (rc == KW_OK) rc = build_band<false>(total, Dh, v, w, st);
    if (rc == KW_OK) rc = solve_mlpg(n_utts, off_dev, total, Dh, w, out_dev, st);
    if (rc != KW_OK) return rc;
    if (mix_dev != nullptr)
        KW_CUDA_CHECK(cudaMemcpyAsync(mix_dev, w.mix, sizeof(int32_t) * total,
                                      cudaMemcpyDeviceToDevice, st));
    return KW_OK;
}

extern "C" int kw_gv_estimate(int n_utts, const int64_t* off_dev, int64_t total_rows, int ld,
                              int col0, int ncols, const double* x_dev, double* utt_var_dev,
                              double* sums_dev, double* mean_dev, double* var_dev, void* stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    KW_REQUIRE(n_utts > 0 && ncols > 0 && col0 >= 0 && col0 + ncols <= ld && total_rows >= 0,
               "kw_gv_estimate: bad sizes");
    KW_REQUIRE((long long)n_utts * ncols < (1LL << 26), "kw_gv_estimate: too many utterances");
    const long long threads = 32LL * n_utts * ncols;
    gv_utt_var_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(
        n_utts, off_dev, ld, col0, ncols, x_dev, utt_var_dev);
    KW_CUDA_CHECK(cudaGetLastError());
    gv_reduce_kernel<<<(ncols + 63) / 64, 64, 0, st>>>(n_utts, off_dev, ncols, utt_var_dev,
                                                      sums_dev, mean_dev, var_dev);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

extern "C" int kw_gv_from_sums(int ncols, const double* sums_dev, double* mean_dev,
                               double* var_dev, void* stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    KW_REQUIRE(ncols > 0, "kw_gv_from_sums: bad sizes");
    gv_from_sums_kernel<<<(ncols + 63) / 64, 64, 0, st>>>(ncols, sums_dev, mean_dev, var_dev);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

extern "C" size_t kw_convert_gv_workspace_bytes(int64_t total_frames, int K, int Dh,
                                                int precision) {
    return carve_convert(CONVERT_GV, total_frames, K, Dh, precision, nullptr).bytes;
}

extern "C" int kw_convert_gv_batch(int n_utts, const int64_t* off_dev, int64_t total,
                                   int max_frames, const double* src_dev, int K, int Dh,
                                   const double* prepared_dev, const double* gv_mean_dev,
                                   const double* gv_var_dev, int gv_iter, double w_traj,
                                   double w_gv, const double* static_src_dev, int static_ld,
                                   double* out_dev, int32_t* mix_dev, double* f_dev,
                                   int32_t* accepted_dev, int precision, void* workspace_dev,
                                   size_t workspace_bytes, void* stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (n_utts == 0 || total == 0) return KW_OK;
    int rc = check_convert("kw_convert_gv_batch", n_utts, total, K, Dh, precision, Dh);
    if (rc != KW_OK) return rc;
    KW_REQUIRE(gv_iter >= 0 && w_traj > 0.0 && w_gv >= 0.0,
               "kw_convert_gv_batch: need gv_iter >= 0, w_traj > 0, w_gv >= 0");
    const int sd = Dh / 3;
    KW_REQUIRE(static_src_dev == nullptr || static_ld >= sd,
               "kw_convert_gv_batch: static_ld %d < static_dim %d", static_ld, sd);
    KW_REQUIRE((long long)n_utts * sd < 2147483647LL,
               "kw_convert_gv_batch: too many utterances for one batch");
    const ConvertWorkspace w = carve_convert(CONVERT_GV, total, K, Dh, precision, workspace_dev);
    if (w.bytes > workspace_bytes)
        return workspace_too_small("kw_convert_gv_batch", w.bytes, workspace_bytes);
    const PreparedView v = view_prepared(const_cast<double*>(prepared_dev), K, Dh);
    rc = hard_sequence(total, src_dev, K, Dh, precision, v, w, st);
    if (rc == KW_OK) rc = utterance_flags(n_utts, off_dev, total, w, st);
    if (rc == KW_OK) rc = build_band<false>(total, Dh, v, w, st);
    if (rc == KW_OK) rc = solve_mlpg(n_utts, off_dev, total, Dh, w, out_dev, st);
    if (rc != KW_OK) return rc;
    if (mix_dev != nullptr)
        KW_CUDA_CHECK(cudaMemcpyAsync(mix_dev, w.mix, sizeof(int32_t) * total,
                                      cudaMemcpyDeviceToDevice, st));
    // the solve factored the bands in place: rebuild them (the band kernel is a pure function of
    // E, the mixture sequence and the flags, all still in the workspace), which moves the same
    // bytes as a saved copy would and keeps the workspace at one band set
    rc = build_band<false>(total, Dh, v, w, st);
    if (rc != KW_OK) return rc;
    GvArgs g;
    g.off = off_dev;
    g.n_utts = n_utts;
    g.sd = sd;
    g.gv_iter = gv_iter;
    g.smem_frames = max(1, min(max_frames, GV_SMEM_FRAMES));
    g.mu = gv_mean_dev;
    g.var = gv_var_dev;
    g.w_traj = w_traj;
    g.w_gv = w_gv;
    g.s = static_src_dev;
    g.s_ld = static_ld;
    g.band = w.band;
    g.step = w.step;
    g.out = out_dev;
    g.total = total;
    g.f_out = f_dev;
    g.acc_out = accepted_dev;
    const size_t smem = sizeof(double) * 6 * (size_t)g.smem_frames;
    KW_CUDA_CHECK(cudaFuncSetAttribute(convert_gv_kernel,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    convert_gv_kernel<<<(unsigned)(n_utts * sd), 32, smem, st>>>(g);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

extern "C" size_t kw_convert_em_workspace_bytes(int64_t total_frames, int K, int Dh,
                                                int precision) {
    return carve_convert(CONVERT_EM, total_frames, K, Dh, precision, nullptr).bytes;
}

extern "C" int kw_convert_em_batch(int n_utts, const int64_t* off_dev, int64_t total,
                                   const double* src_dev, int K, int Dh,
                                   const double* prepared_dev, int em_iter, double* out_dev,
                                   double* loglik_dev, int precision, void* workspace_dev,
                                   size_t workspace_bytes, void* stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    KW_REQUIRE(em_iter >= 1, "kw_convert_em_batch: em_iter must be at least 1, got %d", em_iter);
    KW_REQUIRE(Dh % 3 == 0,
               "kw_convert_em_batch: dim_half %d is not static+delta+delta2 (multiple of 3)", Dh);
    KW_REQUIRE(n_utts >= 0 && total >= 0 && K > 0, "kw_convert_em_batch: bad sizes");
    if (n_utts == 0) return KW_OK;
    if (total == 0) {
        if (loglik_dev != nullptr)
            KW_CUDA_CHECK(cudaMemsetAsync(loglik_dev, 0,
                                          sizeof(double) * (size_t)n_utts * (em_iter + 1), st));
        return KW_OK;
    }
    int rc = check_convert("kw_convert_em_batch", n_utts, total, K, Dh, precision, 2 * Dh);
    if (rc != KW_OK) return rc;
    const ConvertWorkspace w = carve_convert(CONVERT_EM, total, K, Dh, precision, workspace_dev);
    if (w.bytes > workspace_bytes)
        return workspace_too_small("kw_convert_em_batch", w.bytes, workspace_bytes);
    const PreparedView v = view_prepared(const_cast<double*>(prepared_dev), K, Dh);
    rc = hard_sequence(total, src_dev, K, Dh, precision, v, w, st);
    if (rc == KW_OK) rc = utterance_flags(n_utts, off_dev, total, w, st);
    if (rc == KW_OK) rc = build_band<false>(total, Dh, v, w, st);
    if (rc == KW_OK) rc = solve_mlpg(n_utts, off_dev, total, Dh, w, out_dev, st);
    if (rc != KW_OK) return rc;
    const int sd = Dh / 3, D = 2 * Dh;
    convert_em_model_kernel<<<K, 256, 0, st>>>(Dh, v, w.means, w.pc, w.aux);
    KW_CUDA_CHECK(cudaGetLastError());
    KW_CUDA_CHECK(cudaMemcpy2DAsync(w.z, sizeof(double) * D, src_dev, sizeof(double) * Dh,
                                    sizeof(double) * Dh, (size_t)total, cudaMemcpyDeviceToDevice,
                                    st));
    const long long cells = total * sd;
    // E-step at y = out_dev: responsibilities into w.resp, log-normalisers into w.lse and, when
    // asked, their per-utterance sums into column `col` of the trace
    auto estep = [&](int col) -> int {
        convert_em_frames_kernel<<<(unsigned)((cells + 255) / 256), 256, 0, st>>>(
            total, sd, out_dev, w.flags, kDeltaWindows, D, Dh, w.z);
        KW_CUDA_CHECK(cudaGetLastError());
        Posterior post;
        post.resp = w.resp;
        post.lse_frame = w.lse;
        int r = pack_frames(total, w.z, D, precision, w.gmm, st, /*mstep_parts=*/false);
        if (r == KW_OK)
            r = estep_posterior(total, w.z, K, D, w.means, w.pc, w.aux, precision, w.gmm, post, st);
        if (r != KW_OK) return r;
        if (loglik_dev != nullptr) {
            convert_em_loglik_kernel<<<(unsigned)((32LL * n_utts + 255) / 256), 256, 0, st>>>(
                n_utts, off_dev, w.lse, em_iter + 1, col, loglik_dev);
            KW_CUDA_CHECK(cudaGetLastError());
        }
        return KW_OK;
    };
    const size_t soft_smem = sizeof(double) * ((size_t)SOFT_FT * Dh + SOFT_FT);
    for (int it = 0; it < em_iter; ++it) {
        rc = estep(it);
        if (rc != KW_OK) return rc;
        convert_soft_kernel<true><<<(unsigned)((total + SOFT_FT - 1) / SOFT_FT), 96, soft_smem,
                                    st>>>(total, resp_pad(total), K, Dh, src_dev, w.resp, v, w.q,
                                          w.prec);
        KW_CUDA_CHECK(cudaGetLastError());
        rc = build_band<true>(total, Dh, v, w, st);
        if (rc == KW_OK) rc = solve_mlpg(n_utts, off_dev, total, Dh, w, out_dev, st);
        if (rc != KW_OK) return rc;
    }
    if (loglik_dev != nullptr) return estep(em_iter);
    return KW_OK;
}

extern "C" size_t kw_convert_fullcov_prepared_len(int K, int Dh) {
    return view_fullcov(nullptr, K, Dh).len;
}

extern "C" size_t kw_convert_fullcov_prepare_workspace_bytes(int K, int Dh) {
    return carve_fullcov_scratch(K, Dh, nullptr).bytes;
}

extern "C" int kw_convert_fullcov_prepare(int K, int Dh, int diff, const double* covariances_dev,
                                          const double* prepared_dev, double* fullcov_dev,
                                          int32_t* info_dev, void* workspace_dev,
                                          size_t workspace_bytes, void* stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    KW_REQUIRE(K > 0 && Dh > 0, "kw_convert_fullcov_prepare: K, dim_half must be positive");
    KW_REQUIRE(Dh % 3 == 0,
               "kw_convert_fullcov_prepare: dim_half %d is not static+delta+delta2 (multiple of 3)",
               Dh);
    KW_REQUIRE(Dh <= 80, "kw_convert_fullcov_prepare: dim_half %d > 80 unsupported", Dh);
    const PreparedView v = view_prepared(const_cast<double*>(prepared_dev), K, Dh);
    const FullcovScratch w = carve_fullcov_scratch(K, Dh, workspace_dev);
    if (w.bytes > workspace_bytes)
        return workspace_too_small("kw_convert_fullcov_prepare", w.bytes, workspace_bytes);
    const FullcovView f = view_fullcov(fullcov_dev, K, Dh);
    convert_fullcov_sigma_kernel<<<K, 256, 0, st>>>(Dh, diff, covariances_dev, v, w);
    KW_CUDA_CHECK(cudaGetLastError());
    // the precision Cholesky factor of Sigma (info[k] != 0: Sigma_k not positive definite)
    int rc = finalize_launch(K, Dh, 0.0, 0, 0, nullptr, nullptr, w.ones, v.tgt_means, w.sigma,
                             w.pc, w.aux, info_dev, st);
    if (rc != KW_OK) return rc;
    const size_t smem = sizeof(double) * (size_t)Dh * Dh;
    KW_CUDA_CHECK(cudaFuncSetAttribute(convert_fullcov_tables_kernel,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    convert_fullcov_tables_kernel<<<K, 256, smem, st>>>(Dh, v, w.pc, f, kDeltaWindows);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

extern "C" size_t kw_convert_fullcov_workspace_bytes(int64_t total_frames, int K, int Dh,
                                                     int precision) {
    return carve_convert(CONVERT_FULLCOV, total_frames, K, Dh, precision, nullptr).bytes;
}

extern "C" int kw_convert_fullcov_batch(int n_utts, const int64_t* off_dev, int64_t total,
                                        int max_frames, const double* src_dev, int K, int Dh,
                                        const double* prepared_dev, const double* fullcov_dev,
                                        double* out_dev, int32_t* mix_dev, int precision,
                                        void* workspace_dev, size_t workspace_bytes,
                                        void* stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    (void)max_frames;
    if (n_utts == 0 || total == 0) return KW_OK;
    int rc = check_convert("kw_convert_fullcov_batch", n_utts, total, K, Dh, precision, Dh);
    if (rc != KW_OK) return rc;
    const ConvertWorkspace w =
        carve_convert(CONVERT_FULLCOV, total, K, Dh, precision, workspace_dev);
    if (w.bytes > workspace_bytes)
        return workspace_too_small("kw_convert_fullcov_batch", w.bytes, workspace_bytes);
    const FullcovView f = view_fullcov(const_cast<double*>(fullcov_dev), K, Dh);
    // the conditional-mean pass on B^T and h in place of A^T and offset yields g_t = P E_t
    PreparedView vg = view_prepared(const_cast<double*>(prepared_dev), K, Dh);
    vg.at = f.bt;
    vg.offset = f.h;
    rc = hard_sequence(total, src_dev, K, Dh, precision, vg, w, st);
    if (rc == KW_OK) rc = solve_fullcov(n_utts, off_dev, Dh, f, w, out_dev, st);
    if (rc != KW_OK) return rc;
    if (mix_dev != nullptr)
        KW_CUDA_CHECK(cudaMemcpyAsync(mix_dev, w.mix, sizeof(int32_t) * total,
                                      cudaMemcpyDeviceToDevice, st));
    return KW_OK;
}

// ------------------------------------------------------------------------------------------
// Low-delay conversion over n_slots concurrent streams (kw_convert_stream_*).

namespace kw {

constexpr int STREAM_MAX_DELAY = 8192;  // 41 s of 5 ms frames; the push's work grows with it

static int check_stream(const char* fn, int n_slots, int delay, int m, const int32_t* slots_host,
                        int K, int Dh, int precision) {
    KW_REQUIRE(n_slots > 0 && n_slots < (1 << 26), "%s: n_slots %d out of range", fn, n_slots);
    KW_REQUIRE(delay >= 0 && delay <= STREAM_MAX_DELAY, "%s: delay %d is not in [0, %d]", fn,
               delay, STREAM_MAX_DELAY);
    KW_REQUIRE(m >= 0 && m <= n_slots, "%s: m %d is not in [0, n_slots = %d]", fn, m, n_slots);
    KW_REQUIRE(m == 0 || slots_host != nullptr, "%s: slots missing", fn);
    std::vector<char> seen(m > 0 ? (size_t)n_slots : 0, 0);
    for (int i = 0; i < m; ++i) {
        const int s = slots_host[i];
        KW_REQUIRE(s >= 0 && s < n_slots, "%s: slot %d out of range [0, %d)", fn, s, n_slots);
        KW_REQUIRE(!seen[s], "%s: slot %d given twice", fn, s);
        seen[s] = 1;
    }
    return check_convert(fn, 1, 1, K, Dh, precision, Dh);
}

// Source rows, the hard sequence of the m frames, then the step (push) or end kernel.
static int stream_run(const char* fn, bool end, int n_slots, int delay, int m,
                      const int32_t* slots_host, const double* static_dev, int K, int Dh,
                      const double* prepared_dev, double* state_dev, double* out_dev,
                      int64_t* index_dev, int precision, void* workspace_dev,
                      size_t workspace_bytes, cudaStream_t st) {
    int rc = check_stream(fn, n_slots, delay, m, slots_host, K, Dh, precision);
    if (rc != KW_OK) return rc;
    KW_REQUIRE(state_dev != nullptr && out_dev != nullptr && index_dev != nullptr &&
                   (end || static_dev != nullptr),
               "%s: missing device buffer", fn);
    const ConvertWorkspace w = carve_convert(CONVERT_STREAM, m, K, Dh, precision, workspace_dev);
    if (w.bytes > workspace_bytes) return workspace_too_small(fn, w.bytes, workspace_bytes);
    if (m == 0) return KW_OK;
    const int sd = Dh / 3;
    const StreamState s = view_stream_state(state_dev, n_slots, sd, delay);
    const PreparedView v = view_prepared(const_cast<double*>(prepared_dev), K, Dh);
    // pageable or pinned: the call returns once slots_host has been read
    KW_CUDA_CHECK(cudaMemcpyAsync(w.slots, slots_host, sizeof(int) * m, cudaMemcpyHostToDevice, st));
    convert_stream_source_kernel<<<(unsigned)((32LL * m + 127) / 128), 128, 0, st>>>(
        m, sd, end ? 1 : 0, w.slots, static_dev, s, n_slots, w.x, w.jrow);
    KW_CUDA_CHECK(cudaGetLastError());
    rc = hard_sequence(m, w.x, K, Dh, precision, v, w, st);
    if (rc != KW_OK) return rc;
    StreamStepArgs g;
    g.m = m;
    g.n_slots = n_slots;
    g.sd = sd;
    g.Dh = Dh;
    g.delay = delay;
    g.slots = w.slots;
    g.jrow = w.jrow;
    g.mix = w.mix;
    g.E = w.E;
    g.var = v.var;
    g.s = s;
    g.win = kDeltaWindows;
    g.out = out_dev;
    g.index = index_dev;
    const unsigned blocks = (unsigned)(((long long)m * sd + 127) / 128);
    if (end)
        convert_stream_step_kernel<true><<<blocks, 128, 0, st>>>(g);
    else
        convert_stream_step_kernel<false><<<blocks, 128, 0, st>>>(g);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

}  // namespace kw

extern "C" size_t kw_convert_stream_state_len(int n_slots, int Dh, int delay) {
    return view_stream_state(nullptr, n_slots, Dh / 3, delay).len;
}

extern "C" int kw_convert_stream_init(int n_slots, int Dh, int delay, double* state_dev,
                                      void* stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    KW_REQUIRE(n_slots > 0 && n_slots < (1 << 26),
               "kw_convert_stream_init: n_slots %d out of range", n_slots);
    KW_REQUIRE(Dh > 0 && Dh % 3 == 0,
               "kw_convert_stream_init: dim_half %d is not static+delta+delta2 (multiple of 3)", Dh);
    KW_REQUIRE(delay >= 0 && delay <= STREAM_MAX_DELAY,
               "kw_convert_stream_init: delay %d is not in [0, %d]", delay, STREAM_MAX_DELAY);
    KW_REQUIRE(state_dev != nullptr, "kw_convert_stream_init: missing state");
    KW_CUDA_CHECK(cudaMemsetAsync(
        state_dev, 0, sizeof(double) * kw_convert_stream_state_len(n_slots, Dh, delay), st));
    return KW_OK;
}

extern "C" size_t kw_convert_stream_workspace_bytes(int m, int K, int Dh, int delay,
                                                    int precision) {
    (void)delay;
    return carve_convert(CONVERT_STREAM, m, K, Dh, precision, nullptr).bytes;
}

extern "C" int kw_convert_stream_push(int n_slots, int delay, int m, const int32_t* slots_host,
                                      const double* static_dev, int K, int Dh,
                                      const double* prepared_dev, double* state_dev,
                                      double* out_dev, int64_t* frame_dev, int precision,
                                      void* workspace_dev, size_t workspace_bytes, void* stream) {
    return stream_run("kw_convert_stream_push", false, n_slots, delay, m, slots_host, static_dev,
                      K, Dh, prepared_dev, state_dev, out_dev, frame_dev, precision,
                      workspace_dev, workspace_bytes, static_cast<cudaStream_t>(stream));
}

extern "C" int kw_convert_stream_end(int n_slots, int delay, int m, const int32_t* slots_host,
                                     int K, int Dh, const double* prepared_dev, double* state_dev,
                                     double* out_dev, int64_t* count_dev, int precision,
                                     void* workspace_dev, size_t workspace_bytes, void* stream) {
    return stream_run("kw_convert_stream_end", true, n_slots, delay, m, slots_host, nullptr, K,
                      Dh, prepared_dev, state_dev, out_dev, count_dev, precision, workspace_dev,
                      workspace_bytes, static_cast<cudaStream_t>(stream));
}

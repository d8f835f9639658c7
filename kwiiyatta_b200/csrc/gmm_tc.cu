// Tensor-core E-step (precision = 1): the Mahalanobis contraction of the joint-GMM E-step on
// tcgen05 with split-fp16 operands, for sm_100a.
//
//   y_nk = (x_n - mu_k) L_k,   q_nk = || y_nk ||^2      (kwiiyatta/converter/gmm.py:25-26 ->
//   sklearn _estimate_log_gaussian_prob; restated in oracle/gmm_ref.py weighted_log_prob)
//
// Numerics.  X is centred on its column means c and scaled per column by a power of two sigma_d
// so |x'| < 1;  L'_k = diag(sigma) L_k is scaled per output column by a power of two 2^t so its
// largest entry is in [0.5, 1).  Each operand is split  v = hi + lo * 2^-11  with hi = fp16(v),
// lo = fp16((v - hi) * 2^11)  (22 significant bits).  Per (128-frame tile, component):
//   acc  = x_hi . l_lo + x_lo . l_hi          (18 MMAs,  fp32 accumulate in TMEM)
//   acc  = acc * 2^-11 + x_hi . l_hi          (scale-input-d on the first of 9 MMAs)
//   y_j  = acc_j * 2^t_j - (mu_k - c) L_k     (epilogue, fp32; q accumulated in fp64 per 16 columns)
// so the result carries ~2^-22 relative operand error plus the fp32 accumulation of the MMA.
//
// Data movement.  Operands are pre-packed in global memory in the UMMA canonical K-major,
// no-swizzle layout (8 x 8 fp16 core matrices, 128 B each), so a tile is one contiguous block and
// is fetched with a single cp.async.bulk (1-D TMA) onto an mbarrier -- no tensor maps.  The same
// packed X tile is the MN-major operand a tensor-core M-step would need.
//
// Kernel.  Persistent, one CTA per SM, 6 warps: warp 0 = bulk-copy producer, warp 1 = MMA issuer
// (one elected thread), warps 2-5 = epilogue (one TMEM lane quarter each).  Two accumulator stages
// in TMEM (2 x DP columns) overlap the epilogue of component k with the MMAs of k+1.
#include <cuda_fp16.h>

#include <algorithm>

#include "common.cuh"

namespace kw {
namespace tc {

constexpr int TILE_M = 128;
constexpr double LO_SCALE = 2048.0;   // lo parts are stored scaled by 2^11

// ------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug must trap, not hang the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) {
            printf("kwiiyatta_b200: mbarrier wait timed out (block %d thread %d)\n", blockIdx.x,
                   threadIdx.x);
            __trap();
        }
    }
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes,
                                         uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
        ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(dst_smem)),
                 "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols)
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem] * B[smem]; accumulate = 0 overwrites D.
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                         uint32_t idesc, uint32_t accumulate) {
    // executed by the whole (converged) MMA warp; one elected lane issues
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t.reg .b32 r;\n\t"
        "elect.sync r|q, 0xffffffff;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// D = A * B + D * 2^-11  (scale-input-d)
__device__ __forceinline__ void umma_f16_scaled(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                                uint32_t idesc) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t.reg .b32 r;\n\t"
        "elect.sync r|q, 0xffffffff;\n\t"
        "setp.ne.b32 p, 1, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p, 11;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc)
        : "memory");
}
// Variants with the A operand in tensor memory (lanes = rows, 8 columns per 16 fp16 of K).
__device__ __forceinline__ void umma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc,
                                            uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t.reg .b32 r;\n\t"
        "elect.sync r|q, 0xffffffff;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_f16_ts_scaled(uint32_t d_tmem, uint32_t a_tmem,
                                                   uint64_t b_desc, uint32_t idesc) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t.reg .b32 r;\n\t"
        "elect.sync r|q, 0xffffffff;\n\t"
        "setp.ne.b32 p, 1, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p, 11;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc)
        : "memory");
}
// smem (canonical K-major tile, 128 rows x 32 bytes) -> TMEM (128 lanes x 8 columns)
__device__ __forceinline__ void tmem_cp_128x256b(uint32_t taddr, uint64_t s_desc) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t.reg .b32 r;\n\t"
        "elect.sync r|q, 0xffffffff;\n\t"
        "@q tcgen05.cp.cta_group::1.128x256b [%0], %1;\n\t}"
        ::"r"(taddr), "l"(s_desc)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t.reg .b32 r;\n\t"
        "elect.sync r|q, 0xffffffff;\n\t"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
        ::"r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
          "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
          "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ldmatrix (transposed 8x8 b16 tiles) and the legacy warp-level MMA, for the M-step corner block
__device__ __forceinline__ void ldsm4_t(uint32_t addr, uint32_t* r) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr) : "memory");
}
__device__ __forceinline__ void ldsm2_t(uint32_t addr, uint32_t* r) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];"
                 : "=r"(r[0]), "=r"(r[1]) : "r"(addr) : "memory");
}
__device__ __forceinline__ void mma16816(float* d, const uint32_t* a, const uint32_t* b) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, "
                 "{%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
__device__ __forceinline__ void ldsm4(uint32_t addr, uint32_t* r) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr) : "memory");
}
__device__ __forceinline__ void ldsm2(uint32_t addr, uint32_t* r) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];"
                 : "=r"(r[0]), "=r"(r[1]) : "r"(addr) : "memory");
}
// registers -> TMEM: this thread's lane, 8 consecutive 32-bit columns
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t* v) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
        ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]),
          "r"(v[7])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
template <int R> __device__ __forceinline__ void reg_dec() {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(R));
}
template <int R> __device__ __forceinline__ void reg_inc() {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(R));
}

// UMMA shared-memory descriptor, canonical K-major layout without swizzle:
//   element (row r, k-col c) at  (r/8)*SBO + (c/8)*LBO + (r%8)*16 B + (c%8)*2 B.
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes,
                                              uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFFu);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= (uint64_t)1 << 46;  // descriptor version for sm_100
    return d;                // base offset 0, layout type 0 = no swizzle
}
// K-major tile with the 128-byte swizzle (rows of 128 bytes = 64 fp16 of K, 8-row groups 1024
// bytes apart, tile base 1024-byte aligned); a k-step of 16 elements advances the start address
// by 32 bytes inside the swizzle atom.
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFFu);
    d |= (uint64_t)1 << 16;                       // LBO: unused with a swizzled K-major layout
    d |= (uint64_t)(1024 >> 4) << 32;             // SBO: 8 rows x 128 bytes
    d |= (uint64_t)1 << 46;                       // descriptor version for sm_100
    d |= (uint64_t)2 << 61;                       // layout type: SWIZZLE_128B
    return d;
}
// Instruction descriptor: kind::f16, A = B = fp16, D = fp32, both operands K-major.
__host__ __device__ constexpr uint32_t make_idesc(int M, int N) {
    return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// Packed layouts (in halves).  X tile: [part][row group 16][k group DP/8][8][8];
// B (per component): [part][col group DP/8][k group DP/8][8][8].
// The packed X tile is DPB = DP + 16 columns wide: column DP holds the constant 1 (so the M-step
// contraction also yields sum r (x - mu)), the rest of the pad is zero.  Three parts per tile:
// hi, lo * 2^11 (E-step) and lo unscaled (M-step).
__host__ __device__ inline int dpb_of(int DP) { return DP + 16; }
__host__ __device__ inline size_t tile_elems(int DP) { return (size_t)TILE_M * dpb_of(DP); }
constexpr int X_PARTS = 5;   // hi, lo*2^11 (E-step), lo, and K-major hi / lo for the M-step
// L_k is upper triangular, so B[j][d] = L[d][j] vanishes for j < d.  B is stored per 16-wide
// k-step: block ks holds the row groups jg >= 2*ks only, each as two adjacent 8x8 core matrices
// (LBO = 128 B between them, SBO = 256 B between row groups).  Offsets in halves.
__host__ __device__ inline size_t btri_off(int DP, int ks) {
    const int ng = DP / 8;
    return (size_t)128 * (size_t)(ng * ks - ks * (ks - 1));
}
// After the triangular blocks comes one more 16-deep block over ALL column groups: the bias row.
// Its first K index multiplies the column of ones of the packed frames (index DP), so the MMA
// itself subtracts b'_j = sum_d (mu_d - c_d) L[d][j]; the other 15 K indices are zero.
__host__ __device__ inline size_t bbias_off(int DP) { return btri_off(DP, DP / 16); }
__host__ __device__ inline size_t bmat_elems(int DP) { return bbias_off(DP) + (size_t)DP * 16; }

// ------------------------------------------------------------------------------------------
// Column statistics of X: partial sums / min / max per chunk, then centre and power-of-two scale.
// ------------------------------------------------------------------------------------------
// grid = chunks of frames, 256 threads = 8 row workers x 32 column lanes (D <= 160).
__global__ void __launch_bounds__(256)
colstats_partial_kernel(long long N, int D, const double* __restrict__ X,
                        double* __restrict__ partial, long long frames_per_chunk) {
    __shared__ double red[3][8][160];
    const long long n0 = (long long)blockIdx.x * frames_per_chunk;
    const long long n1 = min(N, n0 + frames_per_chunk);
    const int lane = threadIdx.x & 31, rw = threadIdx.x >> 5;
    double s[5], mn[5], mx[5];
#pragma unroll
    for (int q = 0; q < 5; ++q) { s[q] = 0.0; mn[q] = CUDART_INF; mx[q] = -CUDART_INF; }
    for (long long n = n0 + rw; n < n1; n += 8) {
        const double* row = X + n * D;
#pragma unroll
        for (int q = 0; q < 5; ++q) {
            const int d = lane + 32 * q;
            if (d < D) {
                const double v = row[d];
                s[q] += v;
                mn[q] = fmin(mn[q], v);
                mx[q] = fmax(mx[q], v);
            }
        }
    }
#pragma unroll
    for (int q = 0; q < 5; ++q) {
        const int d = lane + 32 * q;
        red[0][rw][d] = s[q];
        red[1][rw][d] = mn[q];
        red[2][rw][d] = mx[q];
    }
    __syncthreads();
    for (int d = threadIdx.x; d < D; d += 256) {
        double ts = 0.0, tmn = CUDART_INF, tmx = -CUDART_INF;
        for (int r = 0; r < 8; ++r) {      // fixed order
            ts += red[0][r][d];
            tmn = fmin(tmn, red[1][r][d]);
            tmx = fmax(tmx, red[2][r][d]);
        }
        double* p = partial + (size_t)blockIdx.x * 3 * D;
        p[d] = ts;
        p[D + d] = tmn;
        p[2 * D + d] = tmx;
    }
}
// xinfo: [centre (DP) | sigma = 2^e (DP)];  one warp per column, 8 columns per CTA
__global__ void __launch_bounds__(256)
colstats_final_kernel(long long N, int D, int DP, int chunks, const double* __restrict__ partial,
                      double* __restrict__ xinfo) {
    const int lane = threadIdx.x & 31;
    const int d = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (d >= DP) return;
    double c = 0.0, sigma = 1.0;
    if (d < D) {
        double s = 0.0, mn = CUDART_INF, mx = -CUDART_INF;
        for (int q = lane; q < chunks; q += 32) {
            const double* p = partial + (size_t)q * 3 * D;
            s += p[d];
            mn = fmin(mn, p[D + d]);
            mx = fmax(mx, p[2 * D + d]);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s += __shfl_xor_sync(0xffffffffu, s, o);
            mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, o));
            mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        }
        c = s / (double)N;
        const double amax = fmax(mx - c, c - mn);
        if (amax > 0.0 && isfinite(amax)) {
            int e;
            frexp(amax, &e);        // amax = m * 2^e, m in [0.5, 1)  ->  amax < 2^e
            sigma = ldexp(1.0, e);
        }
    }
    if (lane == 0) {
        xinfo[d] = c;
        xinfo[DP + d] = sigma;
    }
}

__device__ __forceinline__ void split_store(double v, __half* hi_dst, __half* lo_dst) {
    const __half h = __double2half(v);
    const double r = (v - (double)__half2float(h)) * LO_SCALE;
    *hi_dst = h;
    *lo_dst = __double2half(r);
}

// One CTA per 128-frame tile.
__global__ void pack_x_kernel(long long N, int D, int DP, const double* __restrict__ X,
                              const double* __restrict__ xinfo, __half* __restrict__ xt,
                              int mstep_parts) {
    const long long tile = blockIdx.x;
    const int DPB = dpb_of(DP);
    __half* hi = xt + (size_t)tile * X_PARTS * tile_elems(DP);
    __half* lo_s = hi + tile_elems(DP);
    __half* lo_u = lo_s + tile_elems(DP);
    // M-step operands, K-major with the 128-byte swizzle: per 64-frame tile one 128-byte row per
    // feature (64 frames), its 16-byte chunks (8 frames) XOR-ed with the row number mod 8:
    // element (feature c, frame r) of M-tile r / 64 at  (r/64) 64 DPB + 64 c
    // + 8 (((r%64)/8) ^ (c%8)) + r%8
    __half* hi_k = lo_u + tile_elems(DP);
    __half* lo_k = hi_k + tile_elems(DP);
    const int kg_n = DPB / 8;
    for (int e = threadIdx.x; e < TILE_M * DPB; e += blockDim.x) {
        const int r = e / DPB, c = e - r * DPB;
        const long long n = tile * TILE_M + r;
        double v = 0.0;
        if (n < N && c < D) v = (X[n * D + c] - xinfo[c]) / xinfo[DP + c];
        if (c == DP) v = 1.0;
        // E-step only: a second constant column, 2^-11, multiplies the 2^11-scaled lo part of the
        // bias, so that ONE MMA adds -b' = -(b'_hi + b'_lo) (see pack_l_kernel)
        const bool e_only = c == DP + 1;
        if (e_only) v = 1.0 / LO_SCALE;
        const size_t o = ((size_t)(r >> 3) * kg_n + (c >> 3)) * 64 + (r & 7) * 8 + (c & 7);
        const __half h = __double2half(v);
        const double res = v - (double)__half2float(h);
        hi[o] = h;
        lo_s[o] = __double2half(res * LO_SCALE);
        if (!mstep_parts) continue;          // posterior only (conversion): E-step parts suffice
        lo_u[o] = __double2half(res);
        const size_t ok = (size_t)(r >> 6) * 64 * DPB + (size_t)c * 64 +
                          (size_t)((((r & 63) >> 3) ^ (c & 7)) * 8) + (r & 7);
        hi_k[ok] = e_only ? __double2half(0.0) : h;
        lo_k[ok] = __double2half(res);
    }
}

// One CTA per component: B[j][d] = sigma_d L[d][j] 2^-t (split), the bias row -b'_j 2^-t with
// b'_j = sum_d (mu_d - c_d) L[d][j], and cst = [log|L|, log w, 4^t].  ONE power-of-two scale per
// component: the frames are standardised (|x'| <= 1), so a column of L whose entries are small
// next to the largest one also contributes little to q = |y|^2, and the absolute error bound is
// what matters; with a common scale (and the bias inside the MMA) the epilogue is just
// q = 4^t sum_j acc_j^2, with no per-column vectors to fetch.
// G components share one B operand ("item"): their 8-row groups are interleaved (A g0, B g0,
// A g1, ...), so one MMA of N = G (DP - 16 ks) computes the k-step for all of them and output
// j of component c lands in accumulator column 8 G (j / 8) + 8 c + j % 8 whatever the k-step.
// grid = G * ceil(K / G); components >= K are zero blocks.
// grid (components, PACK_L_SLICES): every slice derives the component's scale (b' and the largest
// entry: one column per thread, loads eight rows at a time), then stores its share of the
// elements, threads running along a row of L so the reads coalesce.  (One CTA per component with
// one load in flight per thread took 78 us of pure memory latency on 64 SMs.)
constexpr int PACK_L_SLICES = 4;
__global__ void __launch_bounds__(256)
pack_l_kernel(int K, int D, int DP, int G, const double* __restrict__ means,
              const double* __restrict__ prec_chol, const double* __restrict__ aux,
              const double* __restrict__ xinfo, __half* __restrict__ bt,
              double* __restrict__ cst) {
    extern __shared__ double bpv[];      // DP: b'_j, then DP: column scales s_d, DP: mu_d - x0_d
    __shared__ double red[256];
    double* sd = bpv + DP;
    double* md = sd + DP;
    const int k = blockIdx.x;
    const int item = k / G, ci = k - item * G;
    const bool real = k < K;
    const double* L = prec_chol + (size_t)(real ? k : 0) * D * D;
    const double* mu = means + (size_t)(real ? k : 0) * D;
    for (int d = threadIdx.x; d < DP; d += blockDim.x) {
        sd[d] = d < D ? xinfo[DP + d] : 0.0;
        md[d] = d < D ? mu[d] - xinfo[d] : 0.0;
    }
    __syncthreads();
    double amax = 0.0;
    for (int j = threadIdx.x; j < DP; j += blockDim.x) {
        double bp = 0.0;
        if (j < D && real) {
            for (int d0 = 0; d0 <= j; d0 += 8) {
                double l[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) l[q] = L[(size_t)min(d0 + q, j) * D + j];   // (clamped: unconditional loads)
                asm volatile("" ::: "memory");      // keep the eight loads together, ahead of their uses
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    if (d0 + q <= j) {
                        amax = fmax(amax, fabs(l[q] * sd[d0 + q]));
                        bp = fma(md[d0 + q], l[q], bp);
                    }
                }
            }
        }
        bpv[j] = bp;
        amax = fmax(amax, fabs(bp));
    }
    red[threadIdx.x] = amax;
    __syncthreads();
    for (int o = blockDim.x >> 1; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) red[threadIdx.x] = fmax(red[threadIdx.x], red[threadIdx.x + o]);
        __syncthreads();
    }
    amax = red[0];
    double scale = 1.0;
    if (amax > 0.0 && isfinite(amax)) {
        int e;
        frexp(amax, &e);
        scale = ldexp(1.0, e);
    }
    const double inv = 1.0 / scale;
    if (threadIdx.x == 0 && real && blockIdx.y == 0) {
        cst[3 * k] = aux[(size_t)k * (D + 2) + D];
        cst[3 * k + 1] = aux[(size_t)k * (D + 2) + D + 1];
        cst[3 * k + 2] = scale * scale;
    }
    __half* hi = bt + (size_t)item * 2 * G * bmat_elems(DP);
    __half* lo = hi + (size_t)G * bmat_elems(DP);
    // element (d, j) = L[d][j] s_d / scale, rows d of this slice, j fastest across the threads
    const int rows = (DP + PACK_L_SLICES - 1) / PACK_L_SLICES;
    const int d_lo = blockIdx.y * rows, d_hi = min(DP, d_lo + rows);
    for (int e0 = d_lo * DP; e0 < d_hi * DP; e0 += 4 * blockDim.x) {
        double v[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int e = e0 + q * blockDim.x + threadIdx.x;
            const int d = e / DP, j = e - d * DP;
            v[q] = (e < d_hi * DP && real && j < D && d <= j) ? L[(size_t)d * D + j] : 0.0;
        }
        asm volatile("" ::: "memory");
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int e = e0 + q * blockDim.x + threadIdx.x;
            if (e >= d_hi * DP) continue;
            const int d = e / DP, j = e - d * DP;
            const int ks = d >> 4, jg = j >> 3;
            if (jg < 2 * ks) continue;             // structurally zero block: not stored
            const size_t o = (size_t)G * btri_off(DP, ks) +
                             ((size_t)(G * (jg - 2 * ks) + ci) * 2 + ((d >> 3) & 1)) * 64 +
                             (j & 7) * 8 + (d & 7);
            split_store(v[q] * sd[d] * inv, hi + o, lo + o);
        }
    }
    if (blockIdx.y == 0) {
        for (int e = threadIdx.x; e < DP * 16; e += blockDim.x) {
            const int j = e >> 4, dd = e & 15, jg = j >> 3;
            // K index 0 (times the column of ones): hi part of -b'_j; K index 1 (times the
            // 2^-11 column): its lo part scaled by 2^11 -- both in the hi operand, one MMA
            const double v = (dd <= 1 && real) ? -bpv[j] * inv : 0.0;
            const size_t o = (size_t)G * bbias_off(DP) +
                             ((size_t)(G * jg + ci) * 2 + ((dd >> 3) & 1)) * 64 + (j & 7) * 8 +
                             (dd & 7);
            const __half h = __double2half(v);
            hi[o] = dd == 0 ? h : __double2half((v - (double)__half2float(h)) * LO_SCALE);
            lo[o] = __double2half(0.0);
        }
    }
}

// ------------------------------------------------------------------------------------------
// The tcgen05 E-step kernel.
// ------------------------------------------------------------------------------------------
struct EstepSmem {
    // byte offsets into dynamic shared memory
    uint32_t a, b_hi, b_lo, scl, cst, qpart, bars, tmem_ptr, total;
};
__host__ __device__ inline EstepSmem estep_smem(int DP, int G) {
    EstepSmem s;
    uint32_t o = 0;
    s.a = o;     o += 2u * TILE_M * dpb_of(DP) * 2;    // hi then lo (scaled)
    s.b_hi = o;  o += 2u * (uint32_t)(G * bmat_elems(DP)) * 2;   // two stages
    s.b_lo = o;  o += 2u * (uint32_t)(G * bmat_elems(DP)) * 2;   // two stages
    s.scl = o;                                          // (unused)
    s.cst = o;   o += 2u * 4 * 8;                      // two stages of [log|L|, log w, 4^t, -]
    s.qpart = o; o += 3u * 4 * TILE_M * 2 * 8;       // [part - 1][item % 4][row][component of the item]
    s.bars = o;  o += 16 * 8;
    s.tmem_ptr = o; o += 16;
    s.total = o;
    return s;
}

// cand[n] of the mode-1 E-step: -1 = the label stands, k >= 0 = compare with component k in
// fp64, REFINE_ALL = take the fp64 argmax over all components
constexpr int32_t REFINE_ALL = -2;

enum { BAR_A_FULL = 0, BAR_A_EMPTY, BAR_BLO_FULL0, BAR_BLO_FULL1, BAR_BLO_EMPTY0, BAR_BLO_EMPTY1,
       BAR_BHI_FULL0, BAR_BHI_FULL1,
       BAR_BHI_EMPTY0, BAR_BHI_EMPTY1, BAR_TM_FULL0, BAR_TM_FULL1, BAR_TM_EMPTY0, BAR_TM_EMPTY1 };

// MODE 0: weighted log-probabilities into wlpT; MODE 1: hard labels into mix and cand.  (The
// mode is a template parameter so that each instantiation keeps only the registers of its own
// epilogue.)
template <int G, int MODE>
__global__ void __launch_bounds__(576, 1)
estep_tc_kernel(long long N, long long Npad, int n_tiles, int K, int D, int DP,
                uint32_t tmem_cols, const __half* __restrict__ xt, const __half* __restrict__ bt,
                const double* __restrict__ cst,
                double* __restrict__ wlpT, int32_t* __restrict__ mix,
                int32_t* __restrict__ cand, double near_tie, int late_release) {
    extern __shared__ __align__(128) unsigned char smem[];
    const EstepSmem L = estep_smem(DP, G);
    __half* a_hi = reinterpret_cast<__half*>(smem + L.a);
    __half* a_lo = a_hi + tile_elems(DP);
    __half* b_hi0 = reinterpret_cast<__half*>(smem + L.b_hi);
    __half* b_lo = reinterpret_cast<__half*>(smem + L.b_lo);
    double* qpart = reinterpret_cast<double*>(smem + L.qpart);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.bars);
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + L.tmem_ptr);

    // warp index through a shuffle so the compiler knows the role branches are warp-uniform
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const uint32_t a_bytes = 2u * TILE_M * dpb_of(DP) * 2;
    // An item = G components sharing one B operand and one accumulator stage (G = 2 when two
    // accumulators fit an MMA's N <= 256: halves the number of MMAs per component).
    const int KI = (K + G - 1) / G;
    const size_t item_elems = (size_t)G * bmat_elems(DP);
    const uint32_t b_bytes = (uint32_t)item_elems * 2;
    const uint32_t acc_w = (uint32_t)(G * DP);
    const uint32_t lbo = 128;
    const uint32_t sbo_a = (uint32_t)(dpb_of(DP) / 8) * 128;
    const int ksteps = DP / 16;
    const uint32_t idesc = make_idesc(TILE_M, G * DP);

    if (threadIdx.x == 0) {
        for (int i = 0; i < 14; ++i) mbar_init(bars + i, (i >= BAR_TM_EMPTY0) ? 16u : 1u);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_ptr, tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    if (warp == 0) {
        // ---------------- producer ----------------
        if (lane == 0) {
            int it = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
                for (int k = 0; k < KI; ++k) {
                    const uint32_t g = (uint32_t)it * KI + k, s = g & 1u, u = g >> 1;
                    const __half* bk = bt + (size_t)k * 2 * item_elems;
                    mbar_wait(bars + BAR_BLO_EMPTY0 + s, (u & 1u) ^ 1u);
                    mbar_expect_tx(bars + BAR_BLO_FULL0 + s, b_bytes);
                    bulk_g2s(b_lo + (size_t)s * item_elems, bk + item_elems, b_bytes,
                             bars + BAR_BLO_FULL0 + s);
                    mbar_wait(bars + BAR_BHI_EMPTY0 + s, (u & 1u) ^ 1u);
                    mbar_expect_tx(bars + BAR_BHI_FULL0 + s, b_bytes);
                    bulk_g2s(b_hi0 + (size_t)s * item_elems, bk, b_bytes,
                             bars + BAR_BHI_FULL0 + s);
                    if (k == 0) {
                        mbar_wait(bars + BAR_A_EMPTY, ((uint32_t)it & 1u) ^ 1u);
                        mbar_expect_tx(bars + BAR_A_FULL, a_bytes);
                        bulk_g2s(a_hi, xt + (size_t)tile * X_PARTS * tile_elems(DP), a_bytes,
                                 bars + BAR_A_FULL);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ---------------- MMA issuer (whole warp converged, one elected lane issues) --------
        {
            // Descriptors are built once; an MMA's operands differ from the base only by a byte
            // offset, i.e. an addition to the (address >> 4) field (the issuing thread is the
            // critical path of the whole kernel, so nothing else is computed per MMA).
            const uint64_t d_a_hi = make_desc(smem_u32(a_hi), lbo, sbo_a);
            const uint64_t d_a_lo = make_desc(smem_u32(a_lo), lbo, sbo_a);
            const uint64_t d_b_lo0 = make_desc(smem_u32(b_lo), 128, 256);
            const uint64_t d_b_lo1 = make_desc(smem_u32(b_lo + item_elems), 128, 256);
            const uint64_t d_b_hi0 = make_desc(smem_u32(b_hi0), 128, 256);
            const uint64_t d_b_hi1 = make_desc(smem_u32(b_hi0 + item_elems), 128, 256);
            constexpr uint64_t KSTEP = 256 >> 4;      // A: 16 fp16 along K = two core matrices
            const uint32_t ta_hi = tmem_base + 2u * acc_w;              // A (hi) after the accumulators
            const uint32_t ta_lo = ta_hi + (uint32_t)DP / 2 + 8;        // hi has the ones k-step too
            const uint64_t bias_off = (uint64_t)(G * bbias_off(DP) * 2) >> 4;   // descriptor address units
            // k-step ks touches output columns [16 ks, DP) only (L_k is triangular):
            //   N = DP - 16 ks, B block at btri_off(ks), accumulator columns from 16 ks.
            const uint32_t ng = (uint32_t)DP / 8;
            const uint32_t Gu = (uint32_t)G;
            int it = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
                for (int k = 0; k < KI; ++k) {
                    const uint32_t g = (uint32_t)it * KI + k, s = g & 1u, u = g >> 1;
                    const uint64_t d_b_hi = s ? d_b_hi1 : d_b_hi0;
                    const uint32_t acc = tmem_base + s * acc_w;
                    if (k == 0) {
                        // stage the frame tile (hi and scaled lo) in tensor memory once per tile:
                        // every MMA of the tile then reads A from TMEM and shared-memory bandwidth
                        // is left to the L_k blocks.  cp and mma execute in issue order.
                        mbar_wait(bars + BAR_A_FULL, (uint32_t)it & 1u);
                        tc_fence_after();
                        for (uint32_t ks = 0; ks < (uint32_t)ksteps; ++ks) {
                            tmem_cp_128x256b(ta_hi + 8 * ks, d_a_hi + ks * KSTEP);
                            tmem_cp_128x256b(ta_lo + 8 * ks, d_a_lo + ks * KSTEP);
                        }
                        // the k-step that holds the column of ones (its lo part is zero)
                        tmem_cp_128x256b(ta_hi + 8 * (uint32_t)ksteps, d_a_hi + (uint64_t)ksteps * KSTEP);
                        umma_commit(bars + BAR_A_EMPTY);
                    }
                    mbar_wait(bars + BAR_TM_EMPTY0 + s, (u & 1u) ^ 1u);
                    mbar_wait(bars + BAR_BLO_FULL0 + s, u & 1u);
                    tc_fence_after();
                    {
                        uint64_t db = s ? d_b_lo1 : d_b_lo0;          // x_hi . l_lo
                        uint32_t id = idesc, cols = (uint32_t)DP;
                        for (uint32_t ks = 0; ks < (uint32_t)ksteps; ++ks) {
                            umma_f16_ts(acc + Gu * 16 * ks, ta_hi + 8 * ks, db, id, ks > 0 ? 1u : 0u);
                            db += (uint64_t)(Gu * (ng - 2 * ks)) * 16;   // next block: G (ng-2ks) 256 B
                            cols -= 16;
                            id = make_idesc(TILE_M, (int)(Gu * cols));
                        }
                    }
                    umma_commit(bars + BAR_BLO_EMPTY0 + s);
                    mbar_wait(bars + BAR_BHI_FULL0 + s, u & 1u);
                    tc_fence_after();
                    {
                        uint64_t db = d_b_hi;          // x_lo . l_hi
                        uint32_t id = idesc, cols = (uint32_t)DP;
                        for (uint32_t ks = 0; ks < (uint32_t)ksteps; ++ks) {
                            umma_f16_ts(acc + Gu * 16 * ks, ta_lo + 8 * ks, db, id, 1u);
                            db += (uint64_t)(Gu * (ng - 2 * ks)) * 16;
                            cols -= 16;
                            id = make_idesc(TILE_M, (int)(Gu * cols));
                        }
                    }
                    {
                        uint64_t db = d_b_hi;          // acc = acc * 2^-11 + x_hi . l_hi
                        umma_f16_ts_scaled(acc, ta_hi, db, idesc);  // ks = 0 spans every column
                        uint32_t cols = (uint32_t)DP;
                        for (uint32_t ks = 1; ks < (uint32_t)ksteps; ++ks) {
                            db += (uint64_t)(Gu * (ng - 2 * (ks - 1))) * 16;
                            cols -= 16;
                            umma_f16_ts(acc + Gu * 16 * ks, ta_hi + 8 * ks, db,
                                        make_idesc(TILE_M, (int)(Gu * cols)), 1u);
                        }
                        // [1, 2^-11] . [-b'_hi, -b'_lo 2^11]: the whole bias in one MMA
                        umma_f16_ts(acc, ta_hi + 8 * (uint32_t)ksteps, d_b_hi + bias_off, idesc, 1u);
                    }
                    umma_commit(bars + BAR_BHI_EMPTY0 + s);
                    umma_commit(bars + BAR_TM_FULL0 + s);
                }
            }
        }
    } else {
        // ---------------- epilogue (warps 2..17) ----------------
        // Four warps per TMEM lane quarter, each takes a quarter of the accumulator columns; the
        // partial q of parts 1..3 goes through shared memory to part 0, which finishes.  (The
        // epilogue, not the MMA, bounds this kernel: more warps = more latency hiding.)
        const uint32_t quarter = (uint32_t)(warp & 3);
        const int part = (warp - 2) >> 2;           // 0..3
        const int row = (int)quarter * 32 + lane;   // TMEM lane = row of the tile
        const int n_chunks = G * ksteps;            // 16-column chunks of an accumulator stage
        const int c_begin = (n_chunks * part) / 4, c_end = (n_chunks * (part + 1)) / 4;
        const double LOG2PI = 1.8378770664093453;
        int it = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
            const long long n = (long long)tile * TILE_M + row;
            double v1 = -CUDART_INF, v2 = -CUDART_INF;
            float v3 = -CUDART_INF_F;     // third best: only compared with near_tie
            int k1 = 0, k2 = -1;
            // per-component constants [log|L|, log w, 4^t] (part 0 finishes the item's
            // components), prefetched one item ahead
            double cc[2][3], nc[2][3];
            auto fetch = [&](int item) {
                if (part == 0) {
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        const int k = min(item * G + c, K - 1);
#pragma unroll
                        for (int e = 0; e < 3; ++e) nc[c][e] = cst[3 * k + e];
                    }
                }
            };
            fetch(0);
            for (int item = 0; item < KI; ++item) {
                const uint32_t g = (uint32_t)it * KI + item, s = g & 1u, u = g >> 1;
#pragma unroll
                for (int c = 0; c < 2; ++c)
#pragma unroll
                    for (int e = 0; e < 3; ++e) cc[c][e] = nc[c][e];
                if (item + 1 < KI) fetch(item + 1);
                mbar_wait(bars + BAR_TM_FULL0 + s, u & 1u);
                tc_fence_after();
                const uint32_t taddr = tmem_base + ((quarter * 32u) << 16) + s * acc_w;
                // with G = 2 a chunk holds 8 columns of the item's first component, then 8 of
                // the second (interleaved row groups of the B operand)
                double qa = 0.0, qb = 0.0;
                // all TMEM loads of this thread's (at most 3) chunks are issued before one wait
                uint32_t v[3][16];
#pragma unroll
                for (int h = 0; h < 3; ++h)
                    if (c_begin + h < c_end) tmem_ld16(taddr + (c_begin + h) * 16, v[h]);
                tmem_ld_wait();
#pragma unroll
                for (int h = 0; h < 3; ++h) {
                    if (c_begin + h >= c_end) break;
                    // the accumulator IS y / 2^t (scale and bias are inside the MMA): sum squares
                    float2 pa = make_float2(0.f, 0.f), pb = make_float2(0.f, 0.f);
#pragma unroll
                    for (int j2 = 0; j2 < 4; ++j2) {
                        const float2 ya = make_float2(__uint_as_float(v[h][2 * j2]),
                                                      __uint_as_float(v[h][2 * j2 + 1]));
                        const float2 yb = make_float2(__uint_as_float(v[h][8 + 2 * j2]),
                                                      __uint_as_float(v[h][8 + 2 * j2 + 1]));
                        pa = __ffma2_rn(ya, ya, pa);
                        pb = __ffma2_rn(yb, yb, pb);
                    }
                    if (G == 2) {
                        qa += (double)(pa.x + pa.y);
                        qb += (double)(pb.x + pb.y);
                    } else {
                        qa += (double)((pa.x + pa.y) + (pb.x + pb.y));
                    }
                }
                tc_fence_before();
                __syncwarp();
                // Every warp frees the accumulator stage as soon as its own columns are in
                // registers, so the MMAs of item g + 2 do not wait for the rest of this item's
                // epilogue (they did: 14 % of the MMA warp's time in EM).  With `late_release`
                // part 0 frees it only after the partial sums (see launch_estep_tc for when).
                if (lane == 0 && (part > 0 || !late_release)) mbar_arrive(bars + BAR_TM_EMPTY0 + s);
                // The partial sums and their named barrier therefore live in a ring of their own,
                // four slots deep: parts 1..3 can only write slot g % 4 after the MMAs of item g,
                // which waited for every warp's arrival for item g - 2 -- and part 0 makes that
                // arrival after it has finished item g - 3, so slots g - 2 .. g are the only ones
                // that can be live.
                const uint32_t q4 = g & 3u;
                if (part > 0) {
                    double* qp = qpart + ((size_t)((part - 1) * 4 + q4) * TILE_M + row) * 2;
                    qp[0] = qa;
                    qp[1] = qb;
                }
                // The only CTA-level synchronisation of an item: parts 1..3 signal that their
                // partial sums are in shared memory (named barrier 3 + slot, they do not wait),
                // part 0 waits for them.
                if (part == 0) asm volatile("bar.sync %0, 512;" ::"r"(3u + q4) : "memory");
                else asm volatile("bar.arrive %0, 512;" ::"r"(3u + q4) : "memory");
                if (part == 0) {
#pragma unroll
                    for (int pp = 0; pp < 3; ++pp) {
                        const double* qp = qpart + ((size_t)(pp * 4 + q4) * TILE_M + row) * 2;
                        qa += qp[0];
                        qb += qp[1];
                    }
                    if (late_release) {      // the stage freed after the partial sums
                        __syncwarp();
                        if (lane == 0) mbar_arrive(bars + BAR_TM_EMPTY0 + s);
                    }
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        const int k = item * G + c;
                        if (c < G && k < K) {
                            const double q = c ? qb : qa;
                            const double wlp =
                                (-0.5 * ((double)D * LOG2PI + q * cc[c][2]) + cc[c][0]) + cc[c][1];
                            if (MODE == 0) {
                                if (n < N) wlpT[(size_t)k * Npad + n] = wlp;
                            } else if (wlp > v1) {
                                v3 = (float)v2; v2 = v1; k2 = k1; v1 = wlp; k1 = k;
                            } else if (wlp > v2) {
                                v3 = (float)v2; v2 = wlp; k2 = k;
                            } else {
                                v3 = fmaxf(v3, (float)wlp);
                            }
                        }
                    }
                }
            }
            if (part == 0 && MODE == 1 && n < N) {
                // to re-check in fp64: the runner-up when only it is within near_tie of the best,
                // every component (REFINE_ALL) when a third one is as well -- with three near the
                // top the tensor cores may have ranked the fp64 best third
                mix[n] = k1;
                cand[n] = (K > 2 && v1 - (double)v3 < near_tie) ? REFINE_ALL
                          : (K > 1 && v1 - v2 < near_tie)         ? k2
                                                                  : -1;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 1) tmem_dealloc(tmem_base, tmem_cols);
}

// Responsibilities from the weighted log-probabilities (component-major), one thread per frame:
// the frame's log-likelihood from one pass (running maximum and rescaled sum; terms more than 46
// below the maximum cannot change a double-precision sum and skip their exp), then
// r = exp(wlp - lse) in place.  A thread walks K values a whole row pitch apart, so the loads are
// issued eight at a time -- with one in flight per thread the kernel was bound by memory latency
// (81 us for 90 MB), not by bandwidth.  lse_frame (may be NULL) receives each frame's lse.
__global__ void __launch_bounds__(128)
lse_kernel(long long N, long long Npad, int K, double* __restrict__ respT,
           double* __restrict__ lse_partial, double* __restrict__ lse_frame) {
    __shared__ double sh[128];
    const long long n = (long long)blockIdx.x * 128 + threadIdx.x;
    double lse = 0.0;
    if (n < N) {
        double* col = respT + n;
        double mx = -CUDART_INF, sum = 0.0;
        for (int k0 = 0; k0 < K; k0 += 8) {
            double v[8];
#pragma unroll
            for (int j = 0; j < 8; ++j)
                v[j] = (k0 + j < K) ? col[(size_t)(k0 + j) * Npad] : -CUDART_INF;
            asm volatile("" ::: "memory");          // eight loads in flight before the first use
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const double dlt = v[j] - mx;
                if (dlt > 0.0) {
                    sum = (dlt < 46.0 ? sum * exp(-dlt) : 0.0) + 1.0;
                    mx = v[j];
                } else if (dlt > -46.0) {
                    sum += exp(dlt);
                }
            }
        }
        lse = log(sum) + mx;
        for (int k0 = 0; k0 < K; k0 += 8) {
            double v[8];
#pragma unroll
            for (int j = 0; j < 8; ++j)
                v[j] = (k0 + j < K) ? col[(size_t)(k0 + j) * Npad] : 0.0;
            asm volatile("" ::: "memory");
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (k0 + j < K) col[(size_t)(k0 + j) * Npad] = exp(v[j] - lse);
        }
        if (lse_frame != nullptr) lse_frame[n] = lse;
    }
    sh[threadIdx.x] = lse;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < 128; ++i) t += sh[i];
        lse_partial[blockIdx.x] = t;
    }
}

// FP64 weighted log-probability of component k (precision Cholesky Lk, aux ak) for the frame
// whose features the warp holds as xr[t] = x[lane + 32 t] (D <= 160).  Lane l owns the columns
// j = l + 32 t of y = x Lk, each summed over ascending d as in the FP64 E-step; the frame's
// features reach the lanes by shuffle and the loads of Lk run ahead of the FMAs.  The sum of
// squares only grows, column block by column block: as soon as the partial value is below
// `floor`, the final one is too, and the function returns -inf.
__device__ double warp_wlp_fp64(int D, const double (&xr)[5], const double* __restrict__ Lk,
                                const double* __restrict__ ak, double floor) {
    const int lane = threadIdx.x & 31;
    const double LOG2PI = 1.8378770664093453;
    double q = 0.0, w = -CUDART_INF;
#pragma unroll
    for (int t = 0; t < 5; ++t) {
        if (32 * t >= D) break;
        const int j = lane + 32 * t, jj = min(j, D - 1);
        double y = 0.0;
#pragma unroll
        for (int tb = 0; tb <= t; ++tb) {
            const double xv = xr[tb];
            const int dn = min(32, D - 32 * tb);
            for (int d0 = 0; d0 < dn; d0 += 16) {
                double l[16];            // sixteen loads in flight before the first FMA
#pragma unroll
                for (int u = 0; u < 16; ++u)
                    l[u] = Lk[(size_t)min(32 * tb + d0 + u, D - 1) * D + jj];
#pragma unroll
                for (int u = 0; u < 16; ++u) {
                    const int d = 32 * tb + d0 + u;
                    const double xd = __shfl_sync(0xffffffffu, xv, (d0 + u) & 31);
                    // L is upper triangular; rows past D (last batch) contribute nothing
                    y = fma(xd, (d <= j && d0 + u < dn) ? l[u] : 0.0, y);
                }
            }
        }
        if (j < D) {
            y -= ak[j];
            q = fma(y, y, q);
        }
        w = (-0.5 * ((double)D * LOG2PI + warp_sum(q)) + ak[D]) + ak[D + 1];
        if (w < floor) return -CUDART_INF;
    }
    return w;
}

// Hard-assignment near-ties: frames whose best components are closer than the tensor-core error
// budget are re-evaluated in FP64 (one warp per frame) -- the best and the runner-up, or all K
// components when a third is close too -- so the mixture sequence equals the FP64 argmax (the
// lowest index on equal FP64 values).  The label's own value comes first, so that the other
// components stop as soon as they fall below it.
__global__ void refine_argmax_kernel(long long N, int K, int D, const double* __restrict__ X,
                                     const double* __restrict__ prec_chol,
                                     const double* __restrict__ aux, int32_t* __restrict__ mix,
                                     const int32_t* __restrict__ cand) {
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
    // a warp looks at 32 frames at a time (one coalesced load of their candidates) and re-checks
    // the flagged ones in turn
    for (long long n0 = warp * 32; n0 < N; n0 += n_warps * 32) {
      const int mine = (n0 + lane < N) ? cand[n0 + lane] : -1;
      unsigned todo = __ballot_sync(0xffffffffu, mine != -1);
      while (todo) {
        const int src = __ffs(todo) - 1;
        todo &= todo - 1;
        const long long n = n0 + src;
        const int kb = __shfl_sync(0xffffffffu, mine, src);
        const int ka = mix[n];
        double xr[5];
#pragma unroll
        for (int t = 0; t < 5; ++t)
            xr[t] = (lane + 32 * t < D) ? X[n * D + lane + 32 * t] : 0.0;
        double wbest = warp_wlp_fp64(D, xr, prec_chol + (size_t)ka * D * D,
                                     aux + (size_t)ka * (D + 2), -CUDART_INF);
        int kbest = ka;
        const bool all = kb == REFINE_ALL;
        for (int c = 0; c < (all ? K : 1); ++c) {
            const int k = all ? c : kb;
            if (k == ka) continue;
            const double w = warp_wlp_fp64(D, xr, prec_chol + (size_t)k * D * D,
                                           aux + (size_t)k * (D + 2), wbest);
            if (w > wbest || (w == wbest && k < kbest)) {
                wbest = w;
                kbest = k;
            }
        }
        if (lane == 0) mix[n] = kbest;
      }
    }
}


// ------------------------------------------------------------------------------------------
// Tensor-core M-step statistics.
//
//   S_k[i][j] = sum_n z_ni x'_nj,   z_ni = r_nk (x'_ni - mu'_ki)        (i, j < DP; x'_{n,DP} = 1)
//
// A = z (generated per (tile, component) by CUDA cores, fp16 hi + lo), B = x' (the packed frames,
// shared by all components); the contraction runs over the frames of a 64-frame tile.  Work item
// = (component, chunk of tiles); the accumulator (rows = features 0..127, columns = features and
// the ones column) is flushed from TMEM after every tile into fp32 registers of the epilogue warps
// (round to nearest, with the tile's weight scale undone) and written as fp32 partials at the end
// of the item, summed in fp64 in a fixed order afterwards.  Rows 128..143 of S (D = 144) are the
// transposes of columns the MMA already produces, except a 16 x 17 corner (second block of the
// partial, rows 112..127).
// ------------------------------------------------------------------------------------------
constexpr int MT = 64;        // frames per M-step tile

struct MstepGeom {
    int DP, DPB, DA;     // DA = rows of the per-component centre table (>= 128)
    int N1, N2;          // widths of the two blocks of a partial (N2 = 0 when DP <= 128)
    int partial_len;     // floats per work item
    bool corner;         // DP == 144: the 16 x 17 block outside the MMA goes to mma.sync warps
};
__host__ __device__ inline MstepGeom mstep_geom(int DP) {
    MstepGeom g;
    g.DP = DP;
    g.DPB = dpb_of(DP);
    g.DA = DP > 128 ? DP : 128;
    g.N1 = g.DPB;
    g.N2 = DP > 128 ? DP + 16 - 128 : 0;
    g.partial_len = 128 * g.N1 + 128 * g.N2;
    g.corner = (DP == 144);
    return g;
}

// mu'_k = fl32((mu_k - c) / sigma) for the generators, one CTA per component.
__global__ void pack_centres_kernel(int K, int D, int DA, const double* __restrict__ centres,
                                    const double* __restrict__ xinfo, int DP,
                                    float* __restrict__ mu32) {
    const int k = blockIdx.x;
    for (int d = threadIdx.x; d < DA; d += blockDim.x) {
        float v = 0.f;
        if (d < D) v = (float)((centres[(size_t)k * D + d] - xinfo[d]) / xinfo[DP + d]);
        mu32[(size_t)k * DA + d] = v;
    }
}

// Per (component, 64-frame tile): everything the M-step kernel needs to know about the weights,
// prepared in parallel over the whole GPU so that its single producer warp only issues copies:
//   flags[k][tile]  1 when some frame of the tile has weight > floor (as fp32, the form the MMAs
//                   see); only such tiles enter the kernel's pipeline
//   wts[k][tile]    WSTRIDE floats: the 64 weights scaled by a power of two into [0.5, 1) at the
//                   tile's maximum, then the inverse scale (one bulk copy puts them in shared memory)
//   tsum[k][tile]   the tile's weight (double; 0 when not flagged): n_k is their fixed-order sum
// One warp per (component, 4 tiles): 8 lanes per tile, 8 consecutive frames per lane.
constexpr int WSTRIDE = MT + 4;
__global__ void __launch_bounds__(256)
mstats_tc_prep_kernel(long long N, long long Npad, int n_mtiles, int n_mt_pad, int K,
                      const double* __restrict__ respT, unsigned char* __restrict__ flags,
                      float* __restrict__ wts, double* __restrict__ tsum, float floor,
                      int tiles_per_chunk, int* __restrict__ item_count) {
    const int lane = threadIdx.x & 31;
    const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int gpk = n_mt_pad / 4;
    const int k = (int)(w / gpk);
    if (k >= K) return;
    const int tile = (int)(w - (long long)k * gpk) * 4 + (lane >> 3);
    const long long n0 = (long long)tile * MT + (lane & 7) * 8;
    double r[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) r[e] = 0.0;
    if (tile < n_mtiles) {
        const double* rp = respT + (size_t)k * Npad + n0;
        if (n0 + 8 <= N) {
            const double2* rp2 = reinterpret_cast<const double2*>(rp);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const double2 v = rp2[e];
                r[2 * e] = v.x;
                r[2 * e + 1] = v.y;
            }
        } else {
#pragma unroll
            for (int e = 0; e < 8; ++e)
                if (n0 + e < N) r[e] = rp[e];
        }
    }
    float f[8];
    float m = 0.f;
    double sum = 0.0;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        f[e] = (float)r[e];
        m = fmaxf(m, f[e]);
        sum += r[e];
    }
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) {
        m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        sum += __shfl_xor_sync(0xffffffffu, sum, o);
    }
    const bool on = m > floor;
    // 2^-ex m in [0.5, 1): power-of-two scale from the exponent bits
    const uint32_t eb = __float_as_uint(m) >> 23;
    const bool normal = eb >= 1u && eb <= 252u;
    const float up = normal ? __uint_as_float((253u - eb) << 23) : 1.f;
    const float inv = normal ? __uint_as_float((eb + 1u) << 23) : 1.f;
    const size_t slot = (size_t)k * n_mt_pad + tile;
    if (on) {
        float4* dst = reinterpret_cast<float4*>(wts + slot * WSTRIDE + (lane & 7) * 8);
        dst[0] = make_float4(f[0] * up, f[1] * up, f[2] * up, f[3] * up);
        dst[1] = make_float4(f[4] * up, f[5] * up, f[6] * up, f[7] * up);
    }
    if ((lane & 7) == 0) {
        flags[slot] = on ? 1 : 0;
        tsum[slot] = on ? sum : 0.0;
        if (on) atomicAdd(item_count + (tile / tiles_per_chunk) * K + k, 1);   // item = chunk K + k
        if (on) *reinterpret_cast<float4*>(wts + slot * WSTRIDE + MT) = make_float4(inv, 0.f, 0.f, 0.f);
    }
}

// Work items (component, chunk of tiles) in the order the persistent CTAs draw them: most tiles
// first.  Frames sorted by dominant component make the items very uneven (0 .. all tiles carry
// weight); drawn in index order the last ones decided the kernel's tail (+12 % on the bench
// workload by list-scheduling the measured counts, tools/time_mstep_real.py).  Counting sort in one
// block; ties in arbitrary order -- the order changes who computes an item, never a result.
__global__ void __launch_bounds__(1024)
mstats_tc_order_kernel(int n_items, const int* __restrict__ item_count, int* __restrict__ order) {
    __shared__ int hist[1024], base[1024];
    hist[threadIdx.x] = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < n_items; i += 1024) atomicAdd(hist + min(item_count[i], 1023), 1);
    __syncthreads();
    {   // base[b] = number of items in bins above b: exclusive scan over descending bins
        __shared__ int wsum[32];
        const int b = 1023 - (int)threadIdx.x, lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
        const int h = hist[b];
        int inc = h;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        if (lane == 31) wsum[wi] = inc;
        __syncthreads();
        if (wi == 0) {
            int t = wsum[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int u = __shfl_up_sync(0xffffffffu, t, o);
                if (lane >= o) t += u;
            }
            wsum[lane] = t;
        }
        __syncthreads();
        base[b] = inc - h + (wi > 0 ? wsum[wi - 1] : 0);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n_items; i += 1024)
        order[atomicAdd(base + min(item_count[i], 1023), 1)] = i;
}

// n_k = fixed-order sum of the tiles' weights; raw[k][partial_len].
__global__ void __launch_bounds__(256)
mstats_tc_nk_kernel(int n_mt_pad, int partial_len, const double* __restrict__ tsum,
                    double* __restrict__ raw) {
    __shared__ double sh[256];
    const int k = blockIdx.x;
    double t = 0.0;
    for (int i = threadIdx.x; i < n_mt_pad; i += 256) t += tsum[(size_t)k * n_mt_pad + i];
    sh[threadIdx.x] = t;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) raw[(size_t)k * (partial_len + 1) + partial_len] = sh[0];
}

// E-step tail for an EM iteration (kw_gmm_estep resp_form 1): from the weighted log-probabilities
// straight to what mstats_tc2_kernel consumes -- the outputs of mstats_tc_prep_kernel -- without
// writing the responsibilities at all.  respT keeps the log-probabilities
// (kw_gmm_normalize_resp turns them into r).
//
// A block owns FB frames (FB / 64 M-step tiles) and stages their K x FB log-probabilities in
// shared memory with one sweep of independent loads; everything after that is on chip:
//   1. two threads per frame: maximum over the components;
//   2. e = exp(wlp - max) once per element (skipped below exp(-46) of the maximum, where a term
//      cannot change a double-precision sum), kept in place, and their sum -> log-likelihood;
//   3. a warp per (tile, share of the components), two frames per lane: r = e / sum, then flag,
//      scaled fp32 weights, inverse scale, tile weight, items' tile counts.
// lse_kernel + mstats_tc_prep_kernel were bound by the FP64 pipe (two exp per element) and two
// more passes over the matrix; this is one exp for the few components near the maximum and one
// read of the matrix.
template <int FB>
__global__ void __launch_bounds__(2 * FB)
lse_prep_kernel(long long N, long long Npad, int K, const double* __restrict__ wlpT,
                double* __restrict__ lse_partial, int n_mt_pad, unsigned char* __restrict__ flags,
                float* __restrict__ wts, double* __restrict__ tsum, float floor,
                int tiles_per_chunk, int* __restrict__ item_count) {
    extern __shared__ double tile_s[];                 // [K][FB]
    __shared__ double mx_s[2][FB], sum_s[2][FB], lse_s[FB];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int fr = threadIdx.x % FB, part = threadIdx.x / FB;     // part 0 / 1: halves of K
    const long long n = (long long)blockIdx.x * FB + fr;
    const int kh = (K + 1) >> 1, k_lo = part * kh, k_hi = min(K, k_lo + kh);
    // global -> shared with cp.async: every load of the block in flight at once, no registers
    // (the compiler would not keep more than five register loads outstanding here)
    if (n < N) {
        const double* col = wlpT + n;
        for (int k = k_lo; k < k_hi; ++k) {
            const unsigned dst = (unsigned)__cvta_generic_to_shared(tile_s + (size_t)k * FB + fr);
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst),
                         "l"(col + (size_t)k * Npad)
                         : "memory");
        }
    } else {
        for (int k = k_lo; k < k_hi; ++k) tile_s[(size_t)k * FB + fr] = -CUDART_INF;
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    double mx = -CUDART_INF;
#pragma unroll 8
    for (int k = k_lo; k < k_hi; ++k) mx = fmax(mx, tile_s[(size_t)k * FB + fr]);
    mx_s[part][fr] = mx;
    __syncthreads();
    mx = fmax(mx_s[0][fr], mx_s[1][fr]);
    double sum = 0.0;
#pragma unroll 4
    for (int k = k_lo; k < k_hi; ++k) {
        const double dlt = tile_s[(size_t)k * FB + fr] - mx;
        const double e = dlt > -46.0 ? exp(dlt) : 0.0;
        tile_s[(size_t)k * FB + fr] = e;
        sum += e;
    }
    sum_s[part][fr] = sum;
    __syncthreads();
    if (part == 0) {
        const double t = sum_s[0][fr] + sum_s[1][fr];
        lse_s[fr] = n < N ? log(t) + mx : 0.0;
        sum_s[0][fr] = n < N ? 1.0 / t : 0.0;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < FB; ++i) t += lse_s[i];
        lse_partial[blockIdx.x] = t;
    }
    constexpr int TPB = FB / MT;                       // tiles per block
    constexpr int SHARE = (2 * FB / 32) / TPB;         // warps per tile
    const int tl = warp % TPB, ws = warp / TPB;
    const int tile = TPB * blockIdx.x + tl;
    const long long n0 = (long long)tile * MT + 2 * lane;
    const bool h0 = n0 < N, h1 = n0 + 1 < N;
    const double i0 = sum_s[0][tl * MT + 2 * lane], i1 = sum_s[0][tl * MT + 2 * lane + 1];
    const int chunk = tile / tiles_per_chunk;
#pragma unroll 2
    for (int k = ws; k < K; k += SHARE) {
        const double2 e = *reinterpret_cast<const double2*>(tile_s + (size_t)k * FB + tl * MT +
                                                            2 * lane);
        const double r0 = h0 ? e.x * i0 : 0.0, r1 = h1 ? e.y * i1 : 0.0;
        const float f0 = (float)r0, f1 = (float)r1;
        const uint32_t mb = __reduce_max_sync(0xffffffffu,
                                              max(__float_as_uint(f0), __float_as_uint(f1)));
        const bool on = __uint_as_float(mb) > floor;
        const size_t slot = (size_t)k * n_mt_pad + tile;
        if (on) {
            double s2 = r0 + r1;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) s2 += __shfl_xor_sync(0xffffffffu, s2, o);
            const uint32_t eb = mb >> 23;
            const bool normal = eb >= 1u && eb <= 252u;
            const float up = normal ? __uint_as_float((253u - eb) << 23) : 1.f;
            *reinterpret_cast<float2*>(wts + slot * WSTRIDE + 2 * lane) =
                make_float2(f0 * up, f1 * up);
            if (lane == 0) {
                const float inv = normal ? __uint_as_float((eb + 1u) << 23) : 1.f;
                *reinterpret_cast<float4*>(wts + slot * WSTRIDE + MT) =
                    make_float4(inv, 0.f, 0.f, 0.f);
                flags[slot] = 1;
                tsum[slot] = s2;
                atomicAdd(item_count + chunk * K + k, 1);
            }
        } else if (lane == 0) {
            flags[slot] = 0;
            tsum[slot] = 0.0;
        }
    }
}

// ------------------------------------------------------------------------------------------
// The M-step kernel: the generated operand lives in TENSOR MEMORY.
//
// Round 1's kernel (git history: mstats_tc_kernel) wrote A = r (x' - mu') to shared memory and the
// MMAs read it back from there; with the packed frames B, the bulk copies and the generators' own
// reads that was 230 KB of shared-memory traffic per (tile, component) against 85 clk x 12 MMAs of
// tensor time, and the shared-memory pipe bounded it (profiles/ncu_r1d_mstats_tc.txt: 49 % LSU
// wavefronts + the MMA operand reads, tensor pipe 38 %; dense case 1.83 ms, now 1.40 ms).  Here
//   * A goes from the generators' registers straight into TMEM (tcgen05.st) and the MMAs take it
//     from there (A-from-TMEM form of tcgen05.mma): no A stores, no A operand reads;
//   * for that a thread must own one FEATURE (TMEM lane) and hold it for consecutive frames (two
//     per 32-bit column), so the packed frames it reads are K-major -- one 128-byte row of 64
//     frames per feature, 128-byte swizzled (pack_x_kernel's hi_k / lo_k parts); one 16-byte load
//     is 8 frames of the thread's feature, and B, the same tile, is a swizzled K-major operand
//   * the shared memory A no longer needs holds a third B stage.
// Rows 128..143 of S (D = 144) are the transposes of columns the big MMA already produces, except
// the 16 x 17 corner, which two mma.sync warps compute as before from a small shared-memory copy
// of those 16 rows of A.  Tiles without weight for the component never enter the pipeline (the
// flags of mstats_tc_prep_kernel / lse_prep_kernel + the producer's ballot over 32 tiles); work
// items are drawn from a global counter, longest first (mstats_tc_order_kernel), and handed to the
// other roles through a 4-slot ring, because frames sorted by dominant component make them very
// uneven.  With dense data the kernel runs into the board's power cap (tools/time_mstep.py; 984 W
// of 1 kW on a B200, commit 1c8d74c); on real posteriors the per-tile hand-offs bound it, as
// measured with per-role wait clocks and switches that turned roles off (commits 1c8d74c to
// 5493bff; the instrumentation is in git history up to a73b842).
// ------------------------------------------------------------------------------------------
constexpr int M2_NB = 3;           // B stages
struct Mstep2Smem {
    uint32_t b_stage, off_b, off_ac, off_rs, off_flags, off_bars, off_tmem, off_corner, total;
};
__host__ __device__ inline Mstep2Smem mstep2_smem(int DP) {
    Mstep2Smem g;
    const int DPB = dpb_of(DP);
    g.b_stage = 2u * MT * DPB * 2;                 // hi + lo
    uint32_t o = 0;
    g.off_b = o;      o += M2_NB * g.b_stage;
    g.off_ac = o;     o += 2u * 2 * 2048;          // corner rows of A: [A stage][hi, lo][2 KB]
    g.off_rs = o;     o += M2_NB * WSTRIDE * 4;     // per B stage: 64 scaled weights + inverse scale
    o = (o + 15u) & ~15u;
    g.off_flags = o;  o += 96;   // item ring[4] | ginv[2] @32 | gflag[2] @48 | pent[3] @64
    g.off_bars = o;   o += 24 * 8;
    g.off_tmem = o;   o += 16;
    g.off_corner = o; o += 2 * 12 * 32 * 4;
    g.total = o;
    return g;
}
enum { M2_B_FULL = 0, M2_B_EMPTY = 3, M2_A_FULL = 6, M2_A_EMPTY = 8, M2_TM_FULL = 10,
       M2_TM_EMPTY = 12, M2_IT_FULL = 14, M2_IT_EMPTY = 18 };

__global__ void __launch_bounds__(640, 1)
mstats_tc2_kernel(long long N, long long Npad, int n_mtiles, int tiles_per_chunk, int n_chunks,
                  int K, int DP, const __half* __restrict__ xt, const float* __restrict__ wts,
                  const float* __restrict__ mu32, float* __restrict__ partial,
                  int* __restrict__ item_counter, const int* __restrict__ item_order,
                  const unsigned char* __restrict__ tflags, int n_mt_pad) {
    extern __shared__ __align__(128) unsigned char smem[];
    const MstepGeom G = mstep_geom(DP);
    const Mstep2Smem L = mstep2_smem(DP);
    unsigned char* b_base = smem + L.off_b;
    unsigned char* ac_base = smem + L.off_ac;
    float* r_s = reinterpret_cast<float*>(smem + L.off_rs);
    volatile int* item_ring = reinterpret_cast<volatile int*>(smem + L.off_flags);          // [4]
    volatile float* ginv = reinterpret_cast<volatile float*>(smem + L.off_flags + 32);     // [2 TMEM stages]
    volatile int* gflag = reinterpret_cast<volatile int*>(smem + L.off_flags + 48);        // [2 TMEM stages]
    volatile int* pent = reinterpret_cast<volatile int*>(smem + L.off_flags + 64);         // [3 B stages]
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.off_bars);
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + L.off_tmem);
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int n_items = K * n_chunks;
    const int DPB = G.DPB;
    const uint32_t part_b = (uint32_t)MT * DPB * 2;      // bytes of one part of a B stage
    const uint32_t acc_cols = (uint32_t)G.N1;            // accumulator stage s at column s * N1
    const uint32_t a_col0 = 2u * acc_cols;               // A stage a: hi at a_col0 + 64 a, lo + 32
    const bool corner = G.corner;

    if (threadIdx.x == 0) {
        for (int i = 0; i < M2_NB; ++i) {
            mbar_init(bars + M2_B_FULL + i, 1);
            mbar_init(bars + M2_B_EMPTY + i, 9 + (corner ? 2 : 0));
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(bars + M2_A_FULL + i, 8);
            mbar_init(bars + M2_A_EMPTY + i, 1 + (corner ? 2 : 0));
            mbar_init(bars + M2_TM_FULL + i, 1);
            mbar_init(bars + M2_TM_EMPTY + i, 8);
        }
        for (int i = 0; i < 4; ++i) {
            mbar_init(bars + M2_IT_FULL + i, 1);
            mbar_init(bars + M2_IT_EMPTY + i, 17 + (corner ? 2 : 0));
        }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_ptr, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    auto next_item = [&](uint32_t idx) -> int {          // consumer side, whole warp
        const uint32_t slot = idx & 3u;
        mbar_wait(bars + M2_IT_FULL + slot, (idx >> 2) & 1u);
        const int it = item_ring[slot];
        __syncwarp();
        if (lane == 0) mbar_arrive(bars + M2_IT_EMPTY + slot);
        return it;
    };
    auto draw_item = [&](uint32_t idx) -> int {          // producer warp
        int it = 0;
        if (lane == 0) {
            const uint32_t slot = idx & 3u;
            mbar_wait(bars + M2_IT_EMPTY + slot, ((idx >> 2) & 1u) ^ 1u);
            it = atomicAdd(item_counter, 1);
            it = it < n_items ? item_order[it] : -1;
            item_ring[slot] = it;
            mbar_arrive(bars + M2_IT_FULL + slot);
        }
        return __shfl_sync(0xffffffffu, it, 0);
    };
    auto item_tiles = [&](int item, int& k, int& t0, int& t1) {
        const int chunk = item / K;
        k = item - chunk * K;
        t0 = chunk * tiles_per_chunk;
        t1 = min(n_mtiles, t0 + tiles_per_chunk);
    };

    if (warp < 4) {
      reg_dec<48>();
      if (warp == 0) {
        // ---------------- producer: K-major packed frames (hi, lo) + the tile's weights -------
        uint32_t g = 0;
        for (uint32_t it_idx = 0;; ++it_idx) {
            const int item = draw_item(it_idx);
            if (item < 0) break;
            int k, t0, t1;
            item_tiles(item, k, t0, t1);
            const unsigned char* fk = tflags + (size_t)k * n_mt_pad;
            const float* wk = wts + (size_t)k * n_mt_pad * WSTRIDE;
            // The item's tiles that carry weight, in order.  This warp is one serial instruction
            // stream per tile, and at ~200 instructions per tile (weights through registers, tile
            // maximum, scale) it was the slowest role of the kernel on real posteriors
            // (per-role wait clocks, commit 5493bff: busy 83 % of the time, the MMA warp
            // waiting).  All of that now happens beforehand in mstats_tc_prep_kernel; here a tile
            // is three bulk copies: packed frames hi, lo and the prepared weights.
            for (int tb = t0; tb < t1; tb += 32) {
                const int tq = tb + lane;
                unsigned mask = __ballot_sync(0xffffffffu, tq < t1 && fk[tq] != 0);
                while (mask) {
                    const int t = tb + __ffs(mask) - 1;
                    mask &= mask - 1;
                    const uint32_t s = g % M2_NB, u = g / M2_NB;
                    mbar_wait(bars + M2_B_EMPTY + s, (u & 1u) ^ 1u);
                    if (lane == 0) {
                        pent[s] = t;
                        mbar_expect_tx(bars + M2_B_FULL + s, 2 * part_b + WSTRIDE * 4);
                        const __half* tile = xt + (size_t)(t >> 1) * X_PARTS * tile_elems(DP) +
                                             3 * tile_elems(DP) + (size_t)(t & 1) * MT * DPB;
                        unsigned char* dst = b_base + s * L.b_stage;
                        bulk_g2s(dst, tile, part_b, bars + M2_B_FULL + s);
                        bulk_g2s(dst + part_b, tile + tile_elems(DP), part_b, bars + M2_B_FULL + s);
                        bulk_g2s(r_s + s * WSTRIDE, wk + (size_t)t * WSTRIDE, WSTRIDE * 4,
                                 bars + M2_B_FULL + s);
                    }
                    __syncwarp();
                    ++g;
                }
            }
            {   // END of the item
                const uint32_t s = g % M2_NB, u = g / M2_NB;
                mbar_wait(bars + M2_B_EMPTY + s, (u & 1u) ^ 1u);
                if (lane == 0) {
                    pent[s] = -1;
                    mbar_arrive(bars + M2_B_FULL + s);
                }
                __syncwarp();
                ++g;
            }
        }
      } else if (warp == 1) {
        // ---------------- MMA issuer: A from TMEM, B K-major from shared memory -----------------
        const uint32_t idesc = make_idesc(128, G.N1);
        // K-major rows of 128 bytes with the 128-byte swizzle
        uint64_t d_b[M2_NB][2];
#pragma unroll
        for (int st = 0; st < M2_NB; ++st)
#pragma unroll
            for (int pt = 0; pt < 2; ++pt)
                d_b[st][pt] = make_desc_sw128(smem_u32(b_base + st * L.b_stage + pt * part_b));
        const uint64_t step_b = 32 >> 4;            // one k-step = 16 frames = 32 bytes of a row
        uint32_t g = 0, f = 0;
        for (uint32_t it_idx = 0;; ++it_idx) {
            const int item = next_item(it_idx);
            if (item < 0) break;
            for (;;) {
                const uint32_t sb = g % M2_NB, ub = g / M2_NB;
                const uint32_t sa = g & 1u, ua = g >> 1;
                const uint32_t ts = f & 1u, tu = f >> 1;
                mbar_wait(bars + M2_B_FULL + sb, ub & 1u);
                const int tt = pent[sb];
                const float tile_inv = r_s[sb * WSTRIDE + MT];
                mbar_wait(bars + M2_TM_EMPTY + ts, (tu & 1u) ^ 1u);
                mbar_wait(bars + M2_A_FULL + sa, ua & 1u);
                tc_fence_after();
                ++g;
                if (tt < 0) {
                    // END: release the stages and close the item with an empty flush group
                    if (lane == 0) {
                        mbar_arrive(bars + M2_A_EMPTY + sa);
                        mbar_arrive(bars + M2_B_EMPTY + sb);
                        gflag[ts] = 2;
                    }
                    __threadfence_block();
                    __syncwarp();
                    umma_commit(bars + M2_TM_FULL + ts);
                    ++f;
                    break;
                }
                const uint32_t acc = tmem_base + ts * acc_cols;
                const uint32_t a_hi = tmem_base + a_col0 + sa * 64u, a_lo = a_hi + 32u;
                const uint64_t b_hi = d_b[sb][0], b_lo = d_b[sb][1];
                // cross passes first (2^-11 of the main term), so only the four A_hi B_hi MMAs
                // truncate the accumulator at full magnitude
#pragma unroll
                for (int pass = 0; pass < 3; ++pass) {
                    const uint32_t ta = (pass == 1) ? a_lo : a_hi;
                    uint64_t db = (pass == 0) ? b_lo : b_hi;
#pragma unroll
                    for (int ks = 0; ks < MT / 16; ++ks) {
                        umma_f16_ts(acc, ta + 8u * ks, db, idesc, (pass > 0 || ks > 0) ? 1u : 0u);
                        db += step_b;
                    }
                }
                umma_commit(bars + M2_A_EMPTY + sa);
                umma_commit(bars + M2_B_EMPTY + sb);
                if (lane == 0) {
                    gflag[ts] = 1;
                    ginv[ts] = tile_inv;
                }
                __threadfence_block();
                __syncwarp();
                umma_commit(bars + M2_TM_FULL + ts);
                ++f;
            }
        }
      } else if (corner) {
        // ---------------- corner warps 2, 3: features 128..143 x columns 128..151 -----------
        // mma.sync m16n8k16 from the K-major tiles: A rows = the 16 corner features (their own
        // small shared-memory copy, written by the generators), B rows = features 128..151 of the
        // packed frames; every 8 x 8 core is an ldmatrix tile as it lies.
        const int cw = warp - 2;
        float* cacc = reinterpret_cast<float*>(smem + L.off_corner) + cw * 12 * 32;
#pragma unroll
        for (int i = 0; i < 12; ++i) cacc[i * 32 + lane] = 0.f;
        const uint32_t mi = (uint32_t)lane >> 3, rr = (uint32_t)lane & 7u;
        // A fragment matrices: (rows 0-7, k 0-7), (rows 8-15, k 0-7), (rows 0-7, k 8-15),
        // (rows 8-15, k 8-15): feature group mi & 1, frame group 2 ks + (mi >> 1)
        const uint32_t la = (((mi & 1u) * 8 + (mi >> 1)) * 8 + rr) * 16;
        // B fragment matrices for column blocks nb, nb + 1: (nb, k 0-7), (nb, k 8-15),
        // (nb + 1, k 0-7), (nb + 1, k 8-15): feature group 16 + nb + (mi >> 1), frame group + (mi & 1)
        // (swizzled rows: feature j = 8 group + rr at j * 128, chunk (frame group ^ rr))
        const uint32_t lb = ((16 + (mi >> 1)) * 8 + rr) * 128;
        const uint32_t lb2 = (18 * 8 + rr) * 128;                       // column block 2 (x2)
        const uint32_t a_s0 = smem_u32(ac_base), b_s0 = smem_u32(b_base);
        float acc[12];
#pragma unroll
        for (int i = 0; i < 12; ++i) acc[i] = 0.f;
        uint32_t g = 0;
        for (uint32_t it_idx = 0;; ++it_idx) {
            const int item = next_item(it_idx);
            if (item < 0) break;
            for (;;) {
                const uint32_t sb = g % M2_NB, ub = g / M2_NB;
                const uint32_t sa = g & 1u, ua = g >> 1;
                mbar_wait(bars + M2_B_FULL + sb, ub & 1u);
                const int tt = pent[sb];
                const float tile_inv = r_s[sb * WSTRIDE + MT];
                mbar_wait(bars + M2_A_FULL + sa, ua & 1u);
                ++g;
                if (tt >= 0) {
                    const uint32_t ab = a_s0 + sa * 4096u + la, bb = b_s0 + sb * L.b_stage;
#pragma unroll
                    for (int kq = 0; kq < MT / 32; ++kq) {
                        const uint32_t ks = (uint32_t)(cw * (MT / 32) + kq);
                        uint32_t ah[4], al[4], bh[6], bl[4];
                        const uint32_t ch = (((2u * ks + (mi & 1u)) ^ rr) << 4);   // swizzled chunk
                        ldsm4(ab + ks * 256u, ah);
                        ldsm4(ab + 2048u + ks * 256u, al);
                        ldsm4(bb + lb + ch, bh);
                        ldsm2(bb + lb2 + ch, bh + 4);
                        ldsm4(bb + part_b + lb + ch, bl);
#pragma unroll
                        for (int nb = 0; nb < 3; ++nb) {
                            mma16816(acc + 4 * nb, al, bh + 2 * nb);
                            // (the ones column of block 2 has no lo part)
                            if (nb < 2) mma16816(acc + 4 * nb, ah, bl + 2 * nb);
                            mma16816(acc + 4 * nb, ah, bh + 2 * nb);
                        }
                    }
                }
                __syncwarp();
                if (lane == 0) {
                    mbar_arrive(bars + M2_A_EMPTY + sa);
                    mbar_arrive(bars + M2_B_EMPTY + sb);
                }
                if (tt >= 0) {
#pragma unroll
                    for (int i = 0; i < 12; ++i) {
                        cacc[i * 32 + lane] = fmaf(acc[i], tile_inv, cacc[i * 32 + lane]);
                        acc[i] = 0.f;
                    }
                }
                if (tt < 0) break;
            }
            asm volatile("bar.sync 3, 64;" ::: "memory");
            if (cw == 1) {
                asm volatile("bar.sync 3, 64;" ::: "memory");    // warp 2 has read our sums
#pragma unroll
                for (int i = 0; i < 12; ++i) cacc[i * 32 + lane] = 0.f;
                continue;
            }
            float* out = partial + (size_t)item * G.partial_len + (size_t)128 * G.N1;
            const int gq = lane >> 2, tq = lane & 3;
#pragma unroll
            for (int nb = 0; nb < 4; ++nb)
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    float2 v = make_float2(0.f, 0.f);
                    if (nb < 3) {
                        v.x = cacc[(4 * nb + 2 * h) * 32 + lane] +
                              cacc[(12 + 4 * nb + 2 * h) * 32 + lane];
                        v.y = cacc[(4 * nb + 2 * h + 1) * 32 + lane] +
                              cacc[(12 + 4 * nb + 2 * h + 1) * 32 + lane];
                        cacc[(4 * nb + 2 * h) * 32 + lane] = 0.f;
                        cacc[(4 * nb + 2 * h + 1) * 32 + lane] = 0.f;
                    }
                    *reinterpret_cast<float2*>(out + (size_t)(112 + gq + 8 * h) * G.N2 + nb * 8 +
                                               2 * tq) = v;
                }
            asm volatile("bar.sync 3, 64;" ::: "memory");
        }
      }
    } else if (warp < 12) {
        reg_dec<88>();
        // ---------------- generators (warps 4..11): A = r (x' - mu') -> TMEM ------------------
        // Thread = feature row i = 32 q + lane of its TMEM lane quarter q = warp % 4; warps 4..7
        // take frame groups 0..3 (k-steps 0, 1), warps 8..11 frame groups 4..7 (k-steps 2, 3).
        // Every thread also converts half a (corner feature, frame group) unit (D > 128).
        const int q = warp & 3, h = (warp - 4) >> 2;
        const int i = 32 * q + lane;
        const bool valid = i < DP;
        const int gt = threadIdx.x - 128;            // 0..255
        // corner unit = (feature 128 + cf, frame group cfg), half a unit (4 frames) per thread so
        // that all eight warps carry the same load
        const int cf = (gt >> 1) & 15, cfg = (gt >> 5) & 7, chalf = gt & 1;
        const bool on_c = corner;
        const uint32_t row_off = (uint32_t)i * 128u, row_x = (uint32_t)(i & 7);
        const uint32_t c_src = (uint32_t)(128 + cf) * 128u +
                               (((uint32_t)cfg ^ (uint32_t)(cf & 7)) << 4) + 8u * (uint32_t)chalf;
        const uint32_t c_dst = ((uint32_t)(cf >> 3) * 8u + (uint32_t)cfg) * 128u +
                               (uint32_t)(cf & 7) * 16u + 8u * (uint32_t)chalf;
        const uint32_t t_lane = tmem_base + (((uint32_t)q * 32u) << 16) + a_col0;
        uint32_t g = 0;
        for (uint32_t it_idx = 0;; ++it_idx) {
            const int item = next_item(it_idx);
            if (item < 0) break;
            int k, t0, t1;
            item_tiles(item, k, t0, t1);
            const float mu_i = valid ? mu32[(size_t)k * G.DA + i] : 0.f;
            const float mu_c = on_c ? mu32[(size_t)k * G.DA + 128 + cf] : 0.f;
            for (;;) {
                const uint32_t sb = g % M2_NB, ub = g / M2_NB;
                const uint32_t sa = g & 1u, ua = g >> 1;
                mbar_wait(bars + M2_B_FULL + sb, ub & 1u);
                const int tt = pent[sb];
                mbar_wait(bars + M2_A_EMPTY + sa, (ua & 1u) ^ 1u);
                tc_fence_after();
                const unsigned char* bh = b_base + sb * L.b_stage;
                const float* rt = r_s + sb * WSTRIDE;
                // 8 frames of one feature: z = r (x' - mu), split into fp16 hi / lo pairs
                auto convert8 = [&](uint32_t off, int fg, float mu, bool live, uint32_t* zh,
                                    uint32_t* zl) {
                    if (!live) {               // feature rows past DP (small D only)
#pragma unroll
                        for (int e = 0; e < 4; ++e) zh[e] = zl[e] = 0u;
                        return;
                    }
                    const uint4 hv = *reinterpret_cast<const uint4*>(bh + off);
                    const uint4 lv = *reinterpret_cast<const uint4*>(bh + part_b + off);
                    const float4 ra = *reinterpret_cast<const float4*>(rt + fg * 8);
                    const float4 rb = *reinterpret_cast<const float4*>(rt + fg * 8 + 4);
                    const float rr8[8] = {ra.x, ra.y, ra.z, ra.w, rb.x, rb.y, rb.z, rb.w};
                    const __half2* hp = reinterpret_cast<const __half2*>(&hv);
                    const __half2* lp = reinterpret_cast<const __half2*>(&lv);
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const float2 xh = __half22float2(hp[e]), xl = __half22float2(lp[e]);
                        const float z0 = rr8[2 * e] * ((xh.x + xl.x) - mu);
                        const float z1 = rr8[2 * e + 1] * ((xh.y + xl.y) - mu);
                        const __half2 zh2 = __floats2half2_rn(z0, z1);
                        const float2 zf = __half22float2(zh2);
                        const __half2 zl2 = __floats2half2_rn(z0 - zf.x, z1 - zf.y);
                        zh[e] = *reinterpret_cast<const uint32_t*>(&zh2);
                        zl[e] = *reinterpret_cast<const uint32_t*>(&zl2);
                    }
                };
                if (tt >= 0) {
#pragma unroll
                    for (int kk = 0; kk < 2; ++kk) {
                        const int ks = 2 * h + kk;
                        uint32_t zh[8], zl[8];
                        convert8(row_off + ((((uint32_t)(2 * ks)) ^ row_x) << 4), 2 * ks, mu_i, valid,
                                 zh, zl);
                        convert8(row_off + ((((uint32_t)(2 * ks + 1)) ^ row_x) << 4), 2 * ks + 1, mu_i,
                                 valid, zh + 4, zl + 4);
                        tmem_st8(t_lane + sa * 64u + 8u * ks, zh);
                        tmem_st8(t_lane + sa * 64u + 32u + 8u * ks, zl);
                    }
                    if (on_c) {
                        // 4 frames of a corner feature
                        const uint2 hv = *reinterpret_cast<const uint2*>(bh + c_src);
                        const uint2 lv = *reinterpret_cast<const uint2*>(bh + part_b + c_src);
                        const float4 ra = *reinterpret_cast<const float4*>(rt + cfg * 8 + chalf * 4);
                        const float rr4[4] = {ra.x, ra.y, ra.z, ra.w};
                        const __half2* hp = reinterpret_cast<const __half2*>(&hv);
                        const __half2* lp = reinterpret_cast<const __half2*>(&lv);
                        uint32_t zh[2], zl[2];
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const float2 xh = __half22float2(hp[e]), xl = __half22float2(lp[e]);
                            const float z0 = rr4[2 * e] * ((xh.x + xl.x) - mu_c);
                            const float z1 = rr4[2 * e + 1] * ((xh.y + xl.y) - mu_c);
                            const __half2 zh2 = __floats2half2_rn(z0, z1);
                            const float2 zf = __half22float2(zh2);
                            const __half2 zl2 = __floats2half2_rn(z0 - zf.x, z1 - zf.y);
                            zh[e] = *reinterpret_cast<const uint32_t*>(&zh2);
                            zl[e] = *reinterpret_cast<const uint32_t*>(&zl2);
                        }
                        unsigned char* dst = ac_base + sa * 4096u + c_dst;
                        *reinterpret_cast<uint2*>(dst) = make_uint2(zh[0], zh[1]);
                        *reinterpret_cast<uint2*>(dst + 2048u) = make_uint2(zl[0], zl[1]);
                    }
                    tmem_st_wait();
                }
                tc_fence_before();
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0) {
                    mbar_arrive(bars + M2_A_FULL + sa);
                    mbar_arrive(bars + M2_B_EMPTY + sb);
                }
                ++g;
                if (tt < 0) break;
            }
        }
    } else {
        reg_inc<128>();
        // ---------------- epilogue (warps 12..19): TMEM -> fp32 registers -> partials -----------
        const uint32_t quarter = (uint32_t)(warp & 3);
        const int half = (warp - 12) >> 2;
        const int row = (int)quarter * 32 + lane;
        const int n16_1 = G.N1 / 16;
        const int c1_begin = half == 0 ? 0 : (n16_1 + 1) / 2;
        const int c1_end = half == 0 ? (n16_1 + 1) / 2 : n16_1;
        float acc[5][16];
        uint32_t f = 0;
        for (uint32_t it_idx = 0;; ++it_idx) {
            const int item = next_item(it_idx);
            if (item < 0) break;
#pragma unroll
            for (int c = 0; c < 5; ++c)
#pragma unroll
                for (int j = 0; j < 16; ++j) acc[c][j] = 0.f;
            for (;;) {
                const uint32_t ts = f & 1u, tu = f >> 1;
                mbar_wait(bars + M2_TM_FULL + ts, tu & 1u);
                tc_fence_after();
                const int fl = gflag[ts];         // bit 0: the group holds data, bit 1: last group
                const bool empty = (fl & 1) == 0;
                const float inv = empty ? 0.f : ginv[ts];
                const float2 inv2 = make_float2(inv, inv);
                const uint32_t tbase = tmem_base + ((quarter * 32u) << 16) + ts * acc_cols;
#pragma unroll
                for (int c = 0; c < 5; ++c) {
                    if (!empty && c1_begin + c < c1_end) {
                        uint32_t v[16];
                        tmem_ld16(tbase + (uint32_t)(c1_begin + c) * 16, v);
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 16; j += 2) {
                            const float2 t = __ffma2_rn(
                                make_float2(__uint_as_float(v[j]), __uint_as_float(v[j + 1])), inv2,
                                make_float2(acc[c][j], acc[c][j + 1]));
                            acc[c][j] = t.x;
                            acc[c][j + 1] = t.y;
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bars + M2_TM_EMPTY + ts);
                ++f;
                if (fl & 2) break;
            }
            float* out = partial + (size_t)item * G.partial_len;
#pragma unroll
            for (int c = 0; c < 5; ++c) {
                if (c1_begin + c < c1_end) {
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        out[(size_t)row * G.N1 + (c1_begin + c) * 16 + j] = acc[c][j];
                }
            }
            if (corner && row < 112) {
                // second block of the partial: only its rows 112..127 carry data (corner warps);
                // the rest is zero so that the shared reduce kernel sums defined values
#pragma unroll
                for (int j = 0; j < 16; ++j)
                    out[(size_t)128 * G.N1 + (size_t)row * G.N2 + half * 16 + j] = 0.f;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// Fixed-order sum of the per-chunk partials: raw[k][e], e < partial_len (n_k, at [partial_len],
// comes from mstats_tc_nk_kernel).
__global__ void mstats_tc_reduce_kernel(int K, int partial_len, int n_chunks,
                                        const float* __restrict__ partial,
                                        double* __restrict__ raw) {
    const int k = blockIdx.y;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < partial_len) {
        // chunks in ascending order, eight loads in flight
        double t = 0.0;
        for (int c0 = 0; c0 < n_chunks; c0 += 8) {
            float v[8];
#pragma unroll
            for (int q = 0; q < 8; ++q)
                v[q] = partial[((size_t)min(c0 + q, n_chunks - 1) * K + k) * partial_len + e];
#pragma unroll
            for (int q = 0; q < 8; ++q)
                if (c0 + q < n_chunks) t += (double)v[q];
        }
        raw[(size_t)k * (partial_len + 1) + e] = t;
    }
}

// Raw sums -> the statistics vector kw_gmm_mstep_finalize expects, centred on centres[k]:
//   n_k,  sum r (x - c_k),  sum r (x - c_k)(x - c_k)^T   (float64).  grid (K, slices).
// `gain` undoes the mean truncation loss of the tensor core's fp32 accumulator: every MMA rounds
// the accumulator toward zero, which on sums of like-signed products (the diagonal, correlated
// pairs, the first moments around a far centre) is a relative loss of about half an ulp per MMA
// at the magnitude the accumulator has reached.  With one tile per flush and the cross passes
// first that is 4 MMAs at 1/4 .. 1 of the tile's sum: -0.7e-7 .. -1.0e-7 relative measured
// (tools/debug_mstats.py), hence gain = 1 + 0.65 * 2^-23.  Sums of mixed-sign products lose less,
// but they are small to begin with.
__global__ void mstats_tc_post_kernel(int K, int D, int DP, const double* __restrict__ raw,
                                      const double* __restrict__ xinfo,
                                      const float* __restrict__ mu32,
                                      const double* __restrict__ centres,
                                      double* __restrict__ stats, double gain) {
    const MstepGeom G = mstep_geom(DP);
    const int k = blockIdx.x;
    const double* sh = raw + (size_t)k * (G.partial_len + 1);
    const double* a1 = sh;
    const double* a2 = sh + 128 * G.N1;
    const double nk = sh[G.partial_len];
    auto sab = [&](int i, int j) -> double {      // needs i < 128 or j >= 128
        if (i < 128) return gain * a1[i * G.N1 + j];
        return gain * a2[(i - (DP - 128)) * G.N2 + (j - 128)];
    };
    const float* muk = mu32 + (size_t)k * G.DA;
    const size_t sb = 1 + (size_t)D + (size_t)D * D;
    double* st = stats + (size_t)k * sb;
    const double* ck = centres + (size_t)k * D;
    // per-feature values every element needs, once per block in shared memory (an element took
    // ~15 dependent global loads before): first moment mc_i, centre of the contraction mu_i,
    // scale s_i, and e_i = effective centre - requested centre in original units
    __shared__ double mc_s[160], mu_s[160], sc_s[160], e_s[160];
    for (int i = threadIdx.x; i < D; i += blockDim.x) {
        const double m = (double)muk[i], si = xinfo[DP + i];
        mc_s[i] = sab(i, DP);
        mu_s[i] = m;
        sc_s[i] = si;
        e_s[i] = (xinfo[i] + si * m) - ck[i];
    }
    __syncthreads();
    auto mc = [&](int i) -> double { return mc_s[i]; };
    auto sc = [&](int i, int j) -> double { return sab(i, j) - mc_s[i] * mu_s[j]; };
    auto eoff = [&](int d) -> double { return e_s[d]; };
    const int tid = blockIdx.y * blockDim.x + threadIdx.x, nthr = gridDim.y * blockDim.x;
    if (tid == 0) st[0] = nk;
    for (int i = tid; i < D; i += nthr)
        st[1 + i] = sc_s[i] * mc(i) + nk * eoff(i);
    for (int e = tid; e < D * D; e += nthr) {
        const int i = e / D, j = e - i * D;
        const bool ok_ij = (i < 128) || (j >= 128), ok_ji = (j < 128) || (i >= 128);
        double v;
        if (ok_ij && ok_ji) v = 0.5 * (sc(i, j) + sc(j, i));
        else if (ok_ij) v = sc(i, j);
        else v = sc(j, i);
        const double si = sc_s[i], sj = sc_s[j];
        const double mi = si * mc(i), mj = sj * mc(j), ei = eoff(i), ej = eoff(j);
        st[1 + D + e] = si * sj * v + mi * ej + ei * mj + nk * ei * ej;
    }
}

}  // namespace tc

constexpr int TC_STAT_CHUNKS = 1184;

// A 64-frame tile enters the tensor-core M-step for a component only if one of its weights
// exceeds this.  What is left out is bounded by floor x (frames in such tiles) per component; on
// the bench workload 28 % of the (component, tile) pairs with any weight above 1e-16 lie below
// 1e-8 and together hold 3.5e-5 frames of weight over all 64 components (n_k ~ 2750 each) -- the
// statistics move by 1.6e-13 of their largest entry, six orders below the rounding of the
// split-fp16 contraction itself (tools/time_mstep_real.py).  The FP64 path keeps 1e-16 per frame.
constexpr float TC_TILE_FLOOR = 1e-8f;
static inline int tc_dp(int D) { return (D + 15) / 16 * 16; }

static int device_sms() {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms;
}

// Number of frame chunks per component for the tensor-core M-step: enough items for a few full
// waves of the persistent grid with the smallest tail.
static int tc_m_chunks(int K, long long n_mtiles) {
    const int sms = 148;
    int best = 1;
    double best_eff = 0.0;
    for (int c = 1; c <= 64; ++c) {
        if ((long long)c > n_mtiles) break;
        const long long items = (long long)K * c;
        if (items < sms && c < 64 && (long long)(c + 1) <= n_mtiles) continue;
        const long long waves = (items + sms - 1) / sms;
        const double eff = (double)items / (double)(waves * sms);
        if (eff > best_eff + 1e-9) { best_eff = eff; best = c; }
        if (items >= 8 * sms) break;
    }
    return best;
}

TcWorkspace carve_tc(Carver& c, long long N, int K, int D) {
    const int DP = tc_dp(D);
    const long long n_tiles = (N + tc::TILE_M - 1) / tc::TILE_M;
    const tc::MstepGeom G = tc::mstep_geom(DP);
    TcWorkspace w;
    w.n_mtiles = (int)(2 * n_tiles);
    w.m_chunks = tc_m_chunks(K, w.n_mtiles);
    w.tiles_per_chunk = (w.n_mtiles + w.m_chunks - 1) / w.m_chunks;
    w.colpartial = c.take<double>((size_t)TC_STAT_CHUNKS * 3 * D);
    w.xinfo = c.take<double>(2 * (size_t)DP);
    w.xt = c.take<__half>((size_t)n_tiles * tc::X_PARTS * tc::tile_elems(DP));
    w.bt = c.take<__half>((size_t)(K + 1) * 2 * tc::bmat_elems(DP));   // (+1: odd K padded to a pair)
    w.sc = c.take<float>((size_t)K * 3 * DP);
    w.cst = c.take<double>(3 * (size_t)K);
    w.lse_partial = c.take<double>(2 * (size_t)n_tiles + 2);
    w.cand = c.take<int32_t>((size_t)N);
    w.mu32 = c.take<float>((size_t)K * G.DA);
    w.mpartial = c.take<float>((size_t)w.m_chunks * K * G.partial_len);
    w.wts = c.take<float>((size_t)K * (size_t)((w.n_mtiles + 3) / 4 * 4) * tc::WSTRIDE);
    w.tsum = c.take<double>((size_t)K * (size_t)((w.n_mtiles + 3) / 4 * 4));
    w.item_counter = c.take<int>(4);
    w.item_count = c.take<int>((size_t)K * w.m_chunks);
    w.item_order = c.take<int>((size_t)K * w.m_chunks);
    w.tflags = c.take<unsigned char>((size_t)K * (size_t)((w.n_mtiles + 3) / 4 * 4));
    w.mraw = c.take<double>((size_t)K * (G.partial_len + 1));
    return w;
}

// Centre, scale, split and tile the frames once per (X, workspace).
int pack_frames(long long N, const double* X, int D, int precision, const GmmWorkspace& gw,
                cudaStream_t st, bool mstep_parts) {
    if (precision != 1) return KW_OK;
    const TcWorkspace& w = gw.tc;
    const int DP = tc_dp(D);
    const long long n_tiles = (N + tc::TILE_M - 1) / tc::TILE_M;
    const long long fpc = (N + TC_STAT_CHUNKS - 1) / TC_STAT_CHUNKS;
    tc::colstats_partial_kernel<<<TC_STAT_CHUNKS, 256, 0, st>>>(N, D, X, w.colpartial, fpc);
    KW_CUDA_CHECK(cudaGetLastError());
    tc::colstats_final_kernel<<<(DP + 7) / 8, 256, 0, st>>>(N, D, DP, TC_STAT_CHUNKS, w.colpartial,
                                                            w.xinfo);
    KW_CUDA_CHECK(cudaGetLastError());
    tc::pack_x_kernel<<<(unsigned)n_tiles, 256, 0, st>>>(N, D, DP, X, w.xinfo, w.xt,
                                                         mstep_parts ? 1 : 0);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

// pack_l_kernel, then estep_tc_kernel<G, mode> over the frames pack_frames left in w: mode 0 writes
// the weighted log-probabilities into resp, mode 1 the labels into mix and the near ties into
// w.cand.
static int launch_estep_tc(long long N, int K, int D, const double* means, const double* pc,
                           const double* aux, const TcWorkspace& w, int mode, double* resp,
                           int32_t* mix, cudaStream_t st) {
    const int DP = tc_dp(D);
    const long long n_tiles = (N + tc::TILE_M - 1) / tc::TILE_M;
    const long long Npad = resp_pad(N);
    // two components per MMA when both accumulators fit N <= 256 and TMEM (DP <= 96)
    const int G = (DP <= 96 && K >= 2) ? 2 : 1;
    const int KI = (K + G - 1) / G;
    tc::pack_l_kernel<<<dim3(KI * G, tc::PACK_L_SLICES), 256, 3 * sizeof(double) * DP, st>>>(K, D, DP, G, means, pc, aux,
                                                                w.xinfo, w.bt, w.cst);
    KW_CUDA_CHECK(cudaGetLastError());
    const tc::EstepSmem L = tc::estep_smem(DP, G);
    uint32_t cols = 32;
    while (cols < 2u * G * DP + DP + 16) cols <<= 1;  // two accumulator stages + the frame tile (hi+ones, lo)
    const int grid = (int)std::min<long long>(n_tiles, device_sms());
    // When the epilogue frees an accumulator stage, measured on one B200 (commit 5844b33): early
    // release takes 4 % off the EM E-step (one component per item, 27 MMAs: the MMA warp was
    // waiting for the stage) and adds 10 % to the conversion posterior (two components per item,
    // a third of the MMA work: the MMAs running further ahead slow the epilogue's TMEM loads).
    // The policy is a kernel argument rather than a constant of the instantiation: folded in at
    // compile time, the late release is hoisted above the partial-sum additions, which frees the
    // stage earlier and made the conversion posterior 9 % slower (B200, 1000 W).
    const int late_release = G == 2 ? 1 : 0;
    auto launch = [&](auto kern) -> int {
        KW_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)L.total));
        kern<<<grid, 576, L.total, st>>>(N, Npad, (int)n_tiles, K, D, DP, cols, w.xt, w.bt, w.cst,
                                         resp, mix, w.cand, 0.05, late_release);
        return KW_OK;
    };
    int rc;
    if (mode == 1)
        rc = (G == 2) ? launch(tc::estep_tc_kernel<2, 1>) : launch(tc::estep_tc_kernel<1, 1>);
    else
        rc = (G == 2) ? launch(tc::estep_tc_kernel<2, 0>) : launch(tc::estep_tc_kernel<1, 0>);
    if (rc != KW_OK) return rc;
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

// Hard labels, with the FP64 re-check of near ties.
int estep_tc_labels(long long N, const double* X, int K, int D, const double* means,
                    const double* pc, const double* aux, const TcWorkspace& w, int32_t* labels,
                    cudaStream_t st) {
    const int rc = launch_estep_tc(N, K, D, means, pc, aux, w, 1, nullptr, labels, st);
    if (rc != KW_OK) return rc;
    tc::refine_argmax_kernel<<<device_sms() * 4, 256, 0, st>>>(N, K, D, X, pc, aux, labels,
                                                               w.cand);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

// The posterior; n_partials: how many log-likelihood partials it leaves in w.lse_partial.
int estep_tc_posterior(long long N, int K, int D, const double* means, const double* pc,
                       const double* aux, const TcWorkspace& w, const Posterior& out,
                       long long& n_partials, cudaStream_t st) {
    const int rc = launch_estep_tc(N, K, D, means, pc, aux, w, 0, out.resp, nullptr, st);
    if (rc != KW_OK) return rc;
    const long long Npad = resp_pad(N);
    unsigned lgrid = (unsigned)((N + 127) / 128);
    if (out.resp_form == 1) {
        // EM iteration: the M-step's inputs straight from the log-probabilities
        KW_CUDA_CHECK(cudaMemsetAsync(w.item_count, 0, sizeof(int) * (size_t)K * w.m_chunks, st));
        const int n_mt_pad = (w.n_mtiles + 3) / 4 * 4;
        // one 64-frame tile per block: 512 K bytes of shared memory, several blocks per SM
        const int sm = K * 64 * (int)sizeof(double);
        // every M-step tile up to n_mt_pad: the M-step reads the flags of all 2 n_tiles tiles (the
        // last one of a final E-tile with at most 64 frames included) and sums the tile weights of
        // all n_mt_pad; a block past N writes "no weight"
        lgrid = (unsigned)n_mt_pad;
        KW_CUDA_CHECK(cudaFuncSetAttribute(tc::lse_prep_kernel<64>,
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, sm));
        tc::lse_prep_kernel<64><<<lgrid, 128, sm, st>>>(
            N, Npad, K, out.resp, w.lse_partial, n_mt_pad, w.tflags, w.wts, w.tsum,
            TC_TILE_FLOOR, w.tiles_per_chunk, w.item_count);
    } else {
        tc::lse_kernel<<<lgrid, 128, 0, st>>>(N, Npad, K, out.resp, w.lse_partial, out.lse_frame);
    }
    KW_CUDA_CHECK(cudaGetLastError());
    n_partials = lgrid;
    return KW_OK;
}

// Weighted log-probabilities left by the posterior with resp_form 1 -> responsibilities, in place.
int normalize_resp_tc(long long N, int K, double* resp, const TcWorkspace& w, cudaStream_t st) {
    tc::lse_kernel<<<(unsigned)((N + 127) / 128), 128, 0, st>>>(N, resp_pad(N), K, resp,
                                                              w.lse_partial, nullptr);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

// M-step statistics on the tensor cores (frames packed by pack_frames).
int mstats_tc(long long N, int K, int D, const double* resp, const double* centres, double* stats,
              const TcWorkspace& w, cudaStream_t st, int resp_form) {
    const int DP = tc_dp(D);
    const tc::MstepGeom G = tc::mstep_geom(DP);
    tc::pack_centres_kernel<<<K, 160, 0, st>>>(K, D, G.DA, centres, w.xinfo, DP, w.mu32);
    KW_CUDA_CHECK(cudaGetLastError());
    const int items = K * w.m_chunks;
    const int grid = std::min(items, device_sms());
    KW_CUDA_CHECK(cudaMemsetAsync(w.item_counter, 0, sizeof(int), st));
    const int n_mt_pad = (w.n_mtiles + 3) / 4 * 4;
    if (resp_form == 0) {
        // (resp_form 1: the posterior left flags, weights, tile sums and item counts in the workspace)
        KW_CUDA_CHECK(cudaMemsetAsync(w.item_count, 0, sizeof(int) * (size_t)items, st));
        const long long warps = (long long)K * (n_mt_pad / 4);
        tc::mstats_tc_prep_kernel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, st>>>(
            N, resp_pad(N), w.n_mtiles, n_mt_pad, K, resp, w.tflags, w.wts, w.tsum,
            TC_TILE_FLOOR, w.tiles_per_chunk, w.item_count);
        KW_CUDA_CHECK(cudaGetLastError());
    }
    tc::mstats_tc_order_kernel<<<1, 1024, 0, st>>>(items, w.item_count, w.item_order);
    KW_CUDA_CHECK(cudaGetLastError());
    const tc::Mstep2Smem L2 = tc::mstep2_smem(DP);
    KW_CUDA_CHECK(cudaFuncSetAttribute(tc::mstats_tc2_kernel,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)L2.total));
    tc::mstats_tc2_kernel<<<grid, 640, L2.total, st>>>(
        N, resp_pad(N), w.n_mtiles, w.tiles_per_chunk, w.m_chunks, K, DP, w.xt, w.wts, w.mu32,
        w.mpartial, w.item_counter, w.item_order, w.tflags, n_mt_pad);
    KW_CUDA_CHECK(cudaGetLastError());
    tc::mstats_tc_reduce_kernel<<<dim3((G.partial_len + 256) / 256, K), 256, 0, st>>>(
        K, G.partial_len, w.m_chunks, w.mpartial, w.mraw);
    KW_CUDA_CHECK(cudaGetLastError());
    tc::mstats_tc_nk_kernel<<<K, 256, 0, st>>>(n_mt_pad, G.partial_len, w.tsum, w.mraw);
    KW_CUDA_CHECK(cudaGetLastError());
    // (a thread's element needs ~15 dependent-latency loads: many small blocks, 2-3 elements each)
    tc::mstats_tc_post_kernel<<<dim3(K, 32), 256, 0, st>>>(K, D, DP, w.mraw, w.xinfo, w.mu32,
                                                          centres, stats, 1.0 + 0.65 / 8388608.0);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

}  // namespace kw

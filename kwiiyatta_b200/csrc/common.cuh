// Shared helpers for the kwiiyatta_b200 CUDA sources (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/kwiiyatta_b200.h"

namespace kw {

void set_error(const char* fmt, ...);

#define KW_CUDA_CHECK(expr)                                                              \
    do {                                                                                 \
        cudaError_t err__ = (expr);                                                      \
        if (err__ != cudaSuccess) {                                                      \
            kw::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(err__),     \
                          __FILE__, __LINE__);                                           \
            return KW_ERR_CUDA;                                                          \
        }                                                                                \
    } while (0)

#define KW_REQUIRE(cond, ...)                                                            \
    do {                                                                                 \
        if (!(cond)) {                                                                   \
            kw::set_error(__VA_ARGS__);                                                  \
            return KW_ERR_INVALID;                                                       \
        }                                                                                \
    } while (0)

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Carves sub-buffers out of a caller-provided workspace.
struct Carver {
    char* base;
    size_t used;
    explicit Carver(void* p) : base(static_cast<char*>(p)), used(0) {}
    template <typename T>
    T* take(size_t count) {
        used = align_up(used, 256);
        T* p = reinterpret_cast<T*>(base + used);
        used += count * sizeof(T);
        return p;
    }
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// gmm.cu internals shared with convert.cu
// lse_frame (mode 0, may be NULL): the per-frame log-normaliser logsumexp_k wlp[n, k]
int estep_fp64(long long N, const double* X, int K, int D, const double* pc, const double* aux,
               double* resp, double* lse_partial, int mode, int32_t* mix, cudaStream_t st,
               double* lse_frame = nullptr);
long long resp_pad(long long n);
void launch_reduce_fixed(const double* in, long long n, double extra, double* out, cudaStream_t st);
// gmm_tc.cu
size_t tc_workspace_bytes(long long N, int K, int D);
int pack_frames_tc(long long N, const double* X, int K, int D, void* workspace,
                   size_t workspace_bytes, cudaStream_t st, bool mstep_parts = true);
int mstats_tc(long long N, const double* X, int K, int D, const double* resp, const double* centres,
              double* stats, void* workspace, size_t workspace_bytes, cudaStream_t st,
              int resp_form = 0);
int normalize_resp_tc(long long N, int K, int D, double* resp, void* workspace,
                      size_t workspace_bytes, cudaStream_t st);
int estep_tc(long long N, const double* X, int K, int D, const double* means, const double* pc,
             const double* aux, double* resp, double* lse_out, int mode, int32_t* mix,
             void* workspace, size_t workspace_bytes, cudaStream_t st, int resp_form = 0,
             double* lse_frame = nullptr);
int mstats_fp64(long long N, const double* X, int K, int D, const double* resp,
                const double* centres, double* partial, double* stats, double resp_floor,
                cudaStream_t st);
int finalize_launch(int K, int D, double reg_covar, int weight_norm, int from_stats,
                    const double* stats, const double* centres, double* weights, double* means,
                    double* cov, double* pc, double* aux, int32_t* info, cudaStream_t st);

}  // namespace kw

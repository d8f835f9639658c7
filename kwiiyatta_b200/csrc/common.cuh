// Shared helpers for the kwiiyatta_b200 CUDA sources (sm_100a only).
#pragma once
#include <cuda_fp16.h>
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

// ---- The GMM layer (gmm.cu, gmm_tc.cu), shared with convert.cu --------------------------------

long long resp_pad(long long n);

constexpr int GMM_MAX_DIM = 144;            // the E-step at both precisions, every tensor-core kernel
constexpr int TC_RESP_FORM1_MAX_K = 384;    // resp_form 1: K x 64 frames of doubles in shared memory
constexpr double RESP_FLOOR = 1e-16;        // the FP64 M-steps skip responsibilities at or below this

// reduce_fixed_kernel: out = { sum of in[0, n) in a fixed order, extra }.
int reduce_fixed(const double* in, long long n, double extra, double* out, cudaStream_t st);

// The tensor-core region of a GMM workspace (precision 1).
struct TcWorkspace {
    double* colpartial;
    double* xinfo;
    __half* xt;
    __half* bt;
    float* sc;
    double* cst;
    double* lse_partial;
    int32_t* cand;
    float* mu32;
    float* mpartial;
    int* item_count;       // tiles with weight per M-step work item
    int* item_order;       // work items, most tiles first
    float* wts;            // per (component, tile): scaled weights + inverse scale (M-step)
    double* tsum;          // per (component, tile): weight of the tile
    int* item_counter;
    unsigned char* tflags;
    double* mraw;
    int m_chunks, tiles_per_chunk, n_mtiles;
};

// What a GMM workspace serves: hard labels only, posteriors (it holds the E-step's log-likelihood
// partials), or the whole fit (the layout of kw_gmm_workspace_bytes).
enum class GmmUse { Labels, Posterior, Fit };

// One layout for (N, K, D, precision), taken from `c`: [FP64 log-likelihood partials (Fit, and
// Posterior at precision 0) | FP64 M-step partials (Fit) | tensor-core region (precision 1)].
// An E-step serves every smaller D from the buffers carved at the largest.
struct GmmWorkspace {
    double* lse_partial;   // the E-step's partials at the workspace's precision (unused for Labels)
    double* partial;       // FP64 M-step partials
    TcWorkspace tc;
};
GmmWorkspace carve_gmm(Carver& c, long long N, int K, int D, int precision, GmmUse use);

// What a posterior E-step writes.  resp (K, resp_pad(N)): responsibilities, or with resp_form 1
// (precision 1; ignored at precision 0) the weighted log-probabilities, which also leaves the
// tensor-core M-step's inputs in the workspace.  total (optional): {sum_n log p(x_n), N}.
// lse_frame (optional, resp_form 0): each frame's log-normaliser logsumexp_k wlp[n, k].
struct Posterior {
    double* resp = nullptr;
    double* total = nullptr;
    double* lse_frame = nullptr;
    int resp_form = 0;
};

// The E-step at either precision, D <= GMM_MAX_DIM.  At precision 1 the frames must have been
// packed into w by pack_frames.  means are read at precision 1 only.
int estep_posterior(long long N, const double* X, int K, int D, const double* means,
                    const double* pc, const double* aux, int precision, const GmmWorkspace& w,
                    const Posterior& out, cudaStream_t st);
// The hard argmax (np.argmax: first max) of every frame into labels.
int estep_labels(long long N, const double* X, int K, int D, const double* means,
                 const double* pc, const double* aux, int precision, const GmmWorkspace& w,
                 int32_t* labels, cudaStream_t st);

// gmm_tc.cu.  Centre, scale, split and tile the frames for the tensor cores (nothing at
// precision 0); mstep_parts = false leaves out the M-step's operands.
int pack_frames(long long N, const double* X, int D, int precision, const GmmWorkspace& w,
                cudaStream_t st, bool mstep_parts = true);
// The tensor-core region (called by carve_gmm only), and the stages behind the calls above.
TcWorkspace carve_tc(Carver& c, long long N, int K, int D);
int estep_tc_posterior(long long N, int K, int D, const double* means, const double* pc,
                       const double* aux, const TcWorkspace& w, const Posterior& out,
                       long long& n_partials, cudaStream_t st);
int estep_tc_labels(long long N, const double* X, int K, int D, const double* means,
                    const double* pc, const double* aux, const TcWorkspace& w, int32_t* labels,
                    cudaStream_t st);
int normalize_resp_tc(long long N, int K, double* resp, const TcWorkspace& w, cudaStream_t st);
int mstats_tc(long long N, int K, int D, const double* resp, const double* centres, double* stats,
              const TcWorkspace& w, cudaStream_t st, int resp_form);
// gmm.cu
int finalize_launch(int K, int D, double reg_covar, int weight_norm, int from_stats,
                    const double* stats, const double* centres, double* weights, double* means,
                    double* cov, double* pc, double* aux, int32_t* info, cudaStream_t st);

}  // namespace kw

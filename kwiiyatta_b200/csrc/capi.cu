// C-ABI plumbing: error reporting, device info, delta features.
#include <cstdarg>
#include <cstring>

#include "common.cuh"

namespace kw {

static thread_local char g_error[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

// delta_features with kwiiyatta's DELTA_WINDOWS (kwiiyatta/converter/delta.py:8-12):
// out[t] = [x[t], -0.5 x[t-1] + 0 x[t] + 0.5 x[t+1], x[t-1] - 2 x[t] + x[t+1]], zero padded
// per utterance, evaluated in np.correlate's left-to-right order.
__global__ void delta_kernel(int n_utts, const int64_t* __restrict__ off, long long total, int dim,
                             const double* __restrict__ in, double* __restrict__ out) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total * dim) return;
    const long long n = e / dim;
    const int d = (int)(e - n * dim);
    // utterance of frame n by binary search
    int lo = 0, hi = n_utts;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (off[mid] <= n) lo = mid; else hi = mid;
    }
    const long long t0 = off[lo], t1 = off[lo + 1];
    const double xc = in[e];
    const double xm = (n - 1 >= t0) ? in[e - dim] : 0.0;
    const double xp = (n + 1 < t1) ? in[e + dim] : 0.0;
    double* o = out + n * 3 * dim;
    o[d] = xc;
    o[dim + d] = __dadd_rn(__dadd_rn(__dmul_rn(-0.5, xm), __dmul_rn(0.0, xc)), __dmul_rn(0.5, xp));
    o[2 * dim + d] = __dadd_rn(__dadd_rn(xm, __dmul_rn(-2.0, xc)), xp);
}

// SPTK mc2b as pysptk.mc2b(mc, alpha) computes it (call site kwiiyatta/filter/mlsa.py:24-29):
// b[M] = mc[M], b[m] = mc[m] - alpha b[m+1]; with zero_power the input's column 0 is taken as 0
// first (the reference removes the power coefficient before the MLSA filter, mlsa.py:23).
// One thread per frame.
__global__ void mc2b_kernel(long long total, int width, double alpha, int zero_power,
                            const double* __restrict__ in, double* __restrict__ out) {
    const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= total) return;
    const double* mc = in + n * width;
    double* b = out + n * width;
    double next = 0.0;
    for (int m = width - 1; m >= 0; --m) {
        const double c = (m == 0 && zero_power) ? 0.0 : mc[m];
        next = (m == width - 1) ? c : __dsub_rn(c, __dmul_rn(alpha, next));
        b[m] = next;
    }
}

}  // namespace kw

using namespace kw;

extern "C" int kw_abi_version(void) { return 3; }

extern "C" const char* kw_last_error(void) { return g_error; }

extern "C" int kw_device_info(int device, int* sm_count, int* cc_major, int* cc_minor,
                              int* clock_khz) {
    cudaDeviceProp prop;
    KW_CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    if (clock_khz) {
        int khz = 0;
        cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, device);
        *clock_khz = khz;
    }
    return KW_OK;
}

extern "C" int kw_delta_features(int n_utts, const int64_t* off_dev, int64_t total_frames, int dim,
                                 const double* in_dev, double* out_dev, void* stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (n_utts == 0 || total_frames == 0) return KW_OK;
    KW_REQUIRE(n_utts > 0 && total_frames > 0 && dim > 0, "kw_delta_features: bad sizes");
    const long long n = (long long)total_frames * dim;
    delta_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n_utts, off_dev, total_frames, dim,
                                                              in_dev, out_dev);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

extern "C" int kw_mc2b(int64_t total_frames, int width, double alpha, int zero_power,
                       const double* mc_dev, double* b_dev, void* stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (total_frames == 0) return KW_OK;
    KW_REQUIRE(total_frames > 0 && width > 0, "kw_mc2b: bad sizes");
    mc2b_kernel<<<(unsigned)((total_frames + 127) / 128), 128, 0, st>>>(
        total_frames, width, alpha, zero_power, mc_dev, b_dev);
    KW_CUDA_CHECK(cudaGetLastError());
    return KW_OK;
}

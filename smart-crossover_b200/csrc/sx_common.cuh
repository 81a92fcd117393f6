// sx_common.cuh -- shared device/host helpers of libsxcross (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/sxcross.h"

namespace sx {

extern int g_last_cuda_error;   // defined in sx_api.cu

inline int cuda_fail(cudaError_t e) {
    g_last_cuda_error = (int)e;
    return SX_ERR_CUDA;
}

#define SX_CUDA(expr)                                        \
    do {                                                     \
        cudaError_t _e = (expr);                             \
        if (_e != cudaSuccess) return ::sx::cuda_fail(_e);   \
    } while (0)

#define SX_LAUNCH_CHECK() SX_CUDA(cudaPeekAtLastError())

// SM count of the current device (148 on a B200: 2 dies x 74 SMs), queried once per device; grids of the
// persistent / cooperative kernels are sized from it.  Defined in sx_api.cu.
int num_sms();

// Lets the current device `dev` access the memory of every other distinct device in devs[0..ndev) (entries equal
// to `dev` are skipped).  SX_ERR_NO_DEVICE when a pair has no peer access.  Defined in sx_api.cu.
int enable_peer_access(int dev, int ndev, const int *devs);

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Bump allocator over a caller-provided workspace.
struct Carver {
    char  *base;
    size_t off = 0;
    explicit Carver(void *p) : base((char *)p) {}
    template <class T> T *take(size_t count) {
        T *r = (T *)(base + off);
        off += align_up(count * sizeof(T), 256);
        return r;
    }
};
inline size_t carve_bytes(size_t count, size_t elem) { return align_up(count * elem, 256); }

// ---- order-preserving images of fp64 ------------------------------------------------
// Unsigned image used by the radix sort: ascending u64 == NumPy's ascending order of the
// doubles, with -0.0 == +0.0 and every NaN last (np.argsort, net_manager.py:184,379).
__host__ __device__ inline unsigned long long f64_to_sort_key(double v) {
#ifdef __CUDA_ARCH__
    unsigned long long b = (unsigned long long)__double_as_longlong(v);
#else
    unsigned long long b; __builtin_memcpy(&b, &v, 8);
#endif
    if ((b << 1) == 0ull) b = 0ull;                                   // -0.0 -> +0.0
    if ((b & 0x7fffffffffffffffull) > 0x7ff0000000000000ull) return ~0ull;   // NaN last
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__host__ __device__ inline double sort_key_to_f64(unsigned long long k) {
    unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
#ifdef __CUDA_ARCH__
    return __longlong_as_double((long long)b);
#else
    double v; __builtin_memcpy(&v, &b, 8); return v;
#endif
}
// Signed image used for atomicMin on reduced costs (no NaN handling needed: NaN never
// compares below -tol, and the min ignores it).
__host__ __device__ inline long long f64_to_min_key(double v) {
    return (long long)(f64_to_sort_key(v) ^ 0x8000000000000000ull);
}
__host__ __device__ inline double min_key_to_f64(long long k) {
    return sort_key_to_f64((unsigned long long)k ^ 0x8000000000000000ull);
}

#ifdef __CUDACC__
__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31u; }

template <class T> __device__ __forceinline__ T warp_min(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        T w = __shfl_xor_sync(0xffffffffu, v, o);
        v = w < v ? w : v;
    }
    return v;
}
template <class T> __device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
#endif

}  // namespace sx

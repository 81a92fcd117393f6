// sx_api.cu -- library-level entry points of libsxcross and the host-buffer pricing call.
#include <math.h>

#include "sx_common.cuh"

namespace sx {
int g_last_cuda_error = 0;

int num_sms() {
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

int enable_peer_access(int dev, int ndev, const int *devs) {
    for (int h = 0; h < ndev; ++h) {
        if (devs[h] == dev) continue;
        int can = 0;
        if (cudaDeviceCanAccessPeer(&can, dev, devs[h]) != cudaSuccess || !can) return SX_ERR_NO_DEVICE;
        cudaError_t e = cudaDeviceEnablePeerAccess(devs[h], 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
        else if (e != cudaSuccess) return cuda_fail(e);
    }
    return SX_OK;
}
}
using namespace sx;

extern "C" int sx_abi_version(void) { return SX_ABI_VERSION; }

extern "C" const char *sx_error_string(int code) {
    switch (code) {
        case SX_OK: return "ok";
        case SX_ERR_INVALID: return "invalid argument";
        case SX_ERR_CUDA: return "CUDA runtime error (see sx_last_cuda_error)";
        case SX_ERR_WORKSPACE: return "workspace too small";
        case SX_ERR_TOO_LARGE: return "problem exceeds the 32-bit arc / node id range of this build";
        case SX_ERR_NOT_SPANNING: return "arcs do not form a spanning tree";
        case SX_ERR_UNALIGNED: return "cost matrix not 16-byte aligned or odd leading dimension";
        case SX_ERR_NO_DEVICE: return "no usable sm_100 device / driver entry point";
        case SX_ERR_PEER_TIMEOUT: return "a peer GPU did not deliver its block in time";
        case SX_ERR_PUSH_ASSERT: return "push phase: no positive flow to push against (reference assertion, tree_BI.py:93-94)";
        default: return "unknown error";
    }
}

extern "C" int sx_last_cuda_error(void) { return g_last_cuda_error; }

extern "C" double sx_key_to_f64(long long key) { return min_key_to_f64(key); }

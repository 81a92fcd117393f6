// sx_exchange.cu -- all-gather of the per-rank pricing result blocks by direct peer stores over
// NVLink / NVSwitch (sm_100a), replacing the NCCL all-gather of the multi-GPU pricing pass.
//
// Every rank owns a symmetric, peer-mapped buffer  [2][G][block_len] int64 slots + [2][G] u64 flags
// + {epoch, done} counters (double-buffered by the parity of a monotonically increasing epoch that
// lives in the buffer itself, so the launch has no per-step argument and can sit in a CUDA graph).
// One launch of G CTAs: CTA p stores this rank's block into slot [parity][rank] of rank p's buffer
// with 128-bit stores, fences at system scope, raises flag [parity][rank] on rank p to `epoch`, and
// then waits until rank p has raised flag [parity][p] in the LOCAL buffer.  When the kernel ends,
// the local slots [parity][0..G) hold all G blocks, the local epoch counter has advanced, and the
// merge kernel (sx_topk_merge with parity_ctr = the epoch counter) consumes them in place.
// 16 KB per rank is pure latency: this costs one kernel (~5 us + NVLink round trip) instead of a
// collective launch.  Ranks run on different GPUs, so the wait never depends on a kernel queued
// behind it on the same device; a bounded spin turns a lost peer into an error code, not a hang.
//
// Double buffering is enough: a rank can only be one epoch ahead of a peer, because finishing epoch
// e + 1 needs that peer's flag for e + 1, which the peer raises after its epoch-e merge (stream order).
#include "sx_ll.cuh"

namespace sx {

__device__ __forceinline__ void st_release_sys(unsigned long long *p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

constexpr int kXcThreads = 256;

__global__ void __launch_bounds__(kXcThreads)
exchange_blocks_kernel(const long long *__restrict__ block, long long block_len, char *const *peer_bufs,
                       int rank, int G, unsigned long long timeout_ns, int *status) {
    const int p = blockIdx.x;                      // peer served by this CTA
    const size_t slots_bytes = (size_t)2 * G * block_len * sizeof(long long);
    char *local = peer_bufs[rank];
    unsigned long long *ctr = reinterpret_cast<unsigned long long *>(local + slots_bytes) + (size_t)2 * G;
    // every CTA reads the counter before any CTA can have finished (it advances only after all G are done)
    const unsigned long long epoch = *reinterpret_cast<volatile unsigned long long *>(ctr) + 1ull;
    const int parity = (int)(epoch & 1ull);
    char *remote = peer_bufs[p];
    long long *dst = reinterpret_cast<long long *>(remote) + ((size_t)parity * G + rank) * block_len;
    // block_len is even and every base is 16-byte aligned: 128-bit stores
    const longlong2 *src2 = reinterpret_cast<const longlong2 *>(block);
    longlong2 *dst2 = reinterpret_cast<longlong2 *>(dst);
    for (long long i = threadIdx.x; i < block_len / 2; i += kXcThreads) dst2[i] = src2[i];
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long *remote_flag =
            reinterpret_cast<unsigned long long *>(remote + slots_bytes) + (size_t)parity * G + rank;
        st_release_sys(remote_flag, epoch);
        const unsigned long long *local_flag =
            reinterpret_cast<const unsigned long long *>(local + slots_bytes) + (size_t)parity * G + p;
        const unsigned long long t0 = global_timer_ns();
        while (ld_acquire_sys(local_flag) < epoch) {
            if (global_timer_ns() - t0 > timeout_ns) { atomicExch(status, SX_ERR_PEER_TIMEOUT); break; }
            __nanosleep(100);
        }
        advance_epoch_when_last(ctr, G, epoch);   // the last CTA to finish
    }
}

// ---- low-latency variant: flag-in-data ("LL") push --------------------------------------------
// Every 8-byte word travels as one 16-byte store {lo32, flag, hi32, flag} with flag = (uint32) epoch,
// so the receiver needs no separate flag, no fence and no second NVLink round trip: it polls each
// slot until both flags show the epoch (8-byte units are written atomically; merge_ll of sx_merge.cuh
// does the polling while it stages the blocks in shared memory).  The kernel only stores, it never waits.
__global__ void __launch_bounds__(kXcThreads)
exchange_push_ll_kernel(const unsigned long long *__restrict__ block, long long block_len, char *const *peer_bufs,
                        int rank, int G) {
    unsigned long long *ctr = ll_counters(peer_bufs[rank], G, block_len);
    const unsigned long long epoch = *reinterpret_cast<volatile unsigned long long *>(ctr) + 1ull;
    uint4 *dst = ll_slot(peer_bufs[blockIdx.x], G, block_len, epoch, rank, 0);
    for (long long i = threadIdx.x; i < block_len; i += kXcThreads) ll_store_slot(dst + i, (unsigned)epoch, block[i]);
    __syncthreads();
    if (threadIdx.x == 0) advance_epoch_when_last(ctr, G, epoch);   // the last CTA to finish
}

}  // namespace sx

using namespace sx;

extern "C" size_t sx_exchange_buffer_bytes(int64_t block_len, int G) {
    if (block_len < 0 || G < 1) return 0;
    return (size_t)2 * G * block_len * 8 + (size_t)2 * G * 8 + 16;
}

extern "C" size_t sx_exchange_epoch_offset(int64_t block_len, int G) {
    if (block_len < 0 || G < 1) return 0;
    return (size_t)2 * G * block_len * 8 + (size_t)2 * G * 8;
}

extern "C" int sx_exchange_blocks(const int64_t *block, int64_t block_len, void *const *peer_bufs_dev, int rank,
                                  int G, int32_t *status_dev, void *stream) {
    if (!block || !peer_bufs_dev || !status_dev || block_len <= 0 || (block_len & 1) || G < 1 || rank < 0 ||
        rank >= G)
        return SX_ERR_INVALID;
    if ((reinterpret_cast<uintptr_t>(block) & 15) != 0) return SX_ERR_UNALIGNED;
    exchange_blocks_kernel<<<G, kXcThreads, 0, (cudaStream_t)stream>>>(
        (const long long *)block, block_len, (char *const *)peer_bufs_dev, rank, G,
        /*timeout_ns=*/10ull * 1000 * 1000 * 1000, status_dev);
    SX_LAUNCH_CHECK();
    return SX_OK;
}

extern "C" size_t sx_exchange_ll_buffer_bytes(int64_t block_len, int G) {
    if (block_len < 0 || G < 1) return 0;
    return (size_t)2 * G * block_len * 16 + 64;
}

extern "C" int sx_exchange_push_ll(const int64_t *block, int64_t block_len, void *const *peer_bufs_dev, int rank,
                                   int G, void *stream) {
    if (!block || !peer_bufs_dev || block_len <= 0 || G < 1 || rank < 0 || rank >= G) return SX_ERR_INVALID;
    exchange_push_ll_kernel<<<G, kXcThreads, 0, (cudaStream_t)stream>>>((const unsigned long long *)block, block_len,
                                                                        (char *const *)peer_bufs_dev, rank, G);
    SX_LAUNCH_CHECK();
    return SX_OK;
}

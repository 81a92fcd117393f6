// sx_ll.cuh -- flag-in-data ("LL") slots of the multi-GPU exchange (sx_exchange.cu, sx_merge.cuh, sx_fused.cu).
// Every 8-byte word travels as one 16-byte store {lo32, flag, hi32, flag} with flag = (uint32) epoch; the
// receiver polls a slot until both flags show the epoch (16-byte stores are single transactions, each
// 8-byte half is written atomically), so no fence, no separate flag and no second NVLink round trip.
// A buffer is [2][G][block_len] slots (the half is the parity of the epoch) followed by the counters
// {push epoch, push CTAs done, merge epoch, merge CTAs done}.
#pragma once
#include "sx_common.cuh"

namespace sx {

__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// slot `idx` of rank r's block in the half of `epoch` of the exchange buffer `buf`
__device__ __forceinline__ uint4 *ll_slot(char *buf, int G, long long block_len, unsigned long long epoch, int r,
                                          long long idx) {
    return reinterpret_cast<uint4 *>(buf) + ((size_t)(epoch & 1ull) * G + r) * block_len + idx;
}
// the counters after the slots
__device__ __forceinline__ unsigned long long *ll_counters(char *buf, int G, long long block_len) {
    return reinterpret_cast<unsigned long long *>(buf + (size_t)2 * G * block_len * 16);
}

// One thread of each of the n_ctas CTAs calls this when its CTA is done with `epoch`; the last one resets the
// done count ctr[1] and publishes the epoch in ctr[0] for the next launch.
__device__ __forceinline__ void advance_epoch_when_last(unsigned long long *ctr, unsigned n_ctas,
                                                        unsigned long long epoch) {
    __threadfence();
    if (atomicAdd(ctr + 1, 1ull) == (unsigned long long)(n_ctas - 1)) {
        ctr[1] = 0ull;
        *reinterpret_cast<volatile unsigned long long *>(ctr) = epoch;
    }
}

__device__ __forceinline__ void ll_store_slot(uint4 *slot, unsigned flag, unsigned long long v) {
    asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(slot), "r"((unsigned)v), "r"(flag),
                 "r"((unsigned)(v >> 32)), "r"(flag)
                 : "memory");
}

__device__ __forceinline__ uint4 ll_load_slot(const uint4 *slot) {
    uint4 w;
    asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(w.x), "=r"(w.y), "=r"(w.z), "=r"(w.w) : "l"(slot) : "memory");
    return w;
}
__device__ __forceinline__ bool ll_ready(const uint4 &w, unsigned flag) { return w.y == flag && w.w == flag; }
__device__ __forceinline__ unsigned long long ll_value(const uint4 &w) {
    return (unsigned long long)w.x | ((unsigned long long)w.z << 32);
}

// Poll one slot until it carries `flag`; false (and v = 0) after timeout_ns.
__device__ __forceinline__ bool ll_poll(const uint4 *slot, unsigned flag, unsigned long long &v,
                                        unsigned long long t0, unsigned long long timeout_ns) {
    for (;;) {
        const uint4 w = ll_load_slot(slot);
        if (ll_ready(w, flag)) { v = ll_value(w); return true; }
        if (global_timer_ns() - t0 > timeout_ns) { v = 0; return false; }
    }
}

}  // namespace sx

// sx_select.cuh -- selection state shared by the pricing kernels (sx_price.cu) and the top-k
// selection (sx_topk.cu).
//
// While a pricing pass streams the arcs, the violators that can still be among the K most
// violating ones are appended to an unordered candidate list, and a two-level histogram over an
// order-preserving 19-bit image of their reduced cost (sign-stripped exponent + 8 mantissa bits,
// 0.4 % relative width per bin) is kept beside it.  Every `kTightenPeriod` appended candidates the
// appending warp scans the histogram for the smallest bin b* whose cumulative count reaches K and
// lowers `bstar` to it: from then on only violators with bin <= b* are appended (the K-th smallest
// reduced cost lies in a bin <= b*, and counts only grow, so the bound stays valid).  The list
// therefore stays O(K log(n/K)) long however many arcs violate, and the final selection
// (sx_topk.cu) is a filter by the final b* plus an all-pairs rank of the few survivors.
#pragma once
#include <stddef.h>

#include "sx_common.cuh"

namespace sx {

constexpr int      kFineBits      = 19;
constexpr unsigned kFineBins      = 1u << kFineBits;          // 524 288 bins, 2 MB
constexpr unsigned kTopBins       = kFineBins / 256;          // 2 048 coarse bins of 256 fine bins
constexpr unsigned kTightenPeriod = 4096;                     // candidates between two tightenings
constexpr int      kSurvCap       = 8192;                     // survivors the all-pairs rank handles

constexpr int kMaxLevels = 16;                                // radix refinement levels of the selection
constexpr int kRefBins   = 2048;                              // 11-bit digits

struct SelState {
    unsigned long long n_cand;       // candidates appended so far (can exceed the buffer capacity)
    unsigned int       bstar;        // only violators with bin <= bstar are appended
    unsigned int       K;            // selection size this pass prunes for
    // header of the pass when the state is one half of a fused pricer (sx_fused.cu); unused otherwise
    sx_price_header    hdr;
    // ---- scratch of the selection kernel (sx_topk.cu), zero at the start of a pass ----
    unsigned int       n_sure;       // elements known to be among the K best (fused kernel: survivors of the filter)
    unsigned int       pad0[3];
    unsigned int       n_list[kMaxLevels + 4];                // boundary-list length per level
    unsigned long long inv_kmin[kMaxLevels + 2];              // ~min key of the level's boundary list
    unsigned long long kmax[kMaxLevels + 2];
    unsigned long long inv_imin[kMaxLevels + 2];              // ~min id
    unsigned long long imax[kMaxLevels + 2];
    unsigned int       hist2[kMaxLevels][kRefBins];
    // ---- histogram of the appended reduced costs (sx_price.cu) ----
    unsigned int       top[kTopBins];
    unsigned int       fine[kFineBins];
};
static_assert(sizeof(SelState) % 16 == 0, "SelState is cleared with 16-byte stores");

// The i-th 16-byte word of a selection state at the start of a pass: everything zero except
// bstar = last bin (no pruning yet), K, and the embedded header's running minimum (= +max).
__host__ __device__ inline uint4 sel_clear_word(size_t i, unsigned K) {
    uint4 z = make_uint4(0u, 0u, 0u, 0u);
    if (i == 0) { z.z = kFineBins - 1u; z.w = K; }                  // n_cand = 0 | bstar | K
    if (i == 1) { z.z = 0xffffffffu; z.w = 0x7fffffffu; }          // hdr.n_violating = 0 | hdr.min_rc_key = INT64_MAX
    return z;
}
static_assert(offsetof(SelState, hdr) == 16, "sel_clear_word assumes the header follows the first 16 bytes");

// (key, id) image of a candidate: key = f64_to_sort_key(rc); (~0, INT64_MAX) is padding.
struct KeyId {
    unsigned long long key;
    long long          id;
};
// L2 load (lists are rewritten by other SMs between grid-wide barriers of one kernel)
__device__ __forceinline__ KeyId ld_keyid(const KeyId *p) {
    const ulonglong2 v = __ldcg(reinterpret_cast<const ulonglong2 *>(p));
    return KeyId{v.x, (long long)v.y};
}
__device__ __forceinline__ bool keyid_less(const KeyId &a, const KeyId &b) {
    return a.key < b.key || (a.key == b.key && a.id < b.id);
}

// bits of sx_price_header.status
constexpr unsigned long long kStatusCandOverflow        = 1ull;   // candidate buffer too small: grow and price again
constexpr unsigned long long kStatusDuplicateCandidates = 2ull;   // one (rc, id) pair repeats too often: selection void
constexpr unsigned long long kStatusKMismatch           = 4ull;   // selection asked for more than the pass pruned for
constexpr unsigned long long kStatusNeedUnfused         = 16ull;  // fused pass could not finish its selection: run the separate kernels
constexpr unsigned long long kStatusNanRc               = 8ull;    // a reduced cost was NaN: not optimal (np.all(rc >= -tol) is False)

// Monotone (non-strict) 19-bit image of a reduced cost: a < b  =>  bin(a) <= bin(b).
// Negative values (every violator when tol >= 0) use the full resolution; anything >= +0 clamps
// into the last bin.
__device__ __forceinline__ unsigned cand_bin(double rc) {
    const unsigned long long k = f64_to_sort_key(rc) >> (64 - 1 - kFineBits);   // sign + 19 bits
    return k < (unsigned long long)kFineBins ? (unsigned)k : kFineBins - 1u;
}

__device__ __forceinline__ unsigned ld_relaxed_u32(const unsigned *p) {
    unsigned v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint4 ld_relaxed_v4(const unsigned *p) {
    uint4 v;
    asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
    return v;
}

// Position of rank `need` in N per-lane counts v[] whose warp-wide inclusive scan crosses `need` in
// this lane: q = first index with before + v[0..q] >= need, before is advanced to the sum below q.
// Static indexing only (v stays in registers).
template <int N>
__device__ __forceinline__ int find_in_lane(const unsigned (&v)[N], unsigned need, unsigned &before) {
    int q = -1;
#pragma unroll
    for (int r = 0; r < N; ++r) {
        if (q < 0) {
            if (before + v[r] >= need) q = r; else before += v[r];
        }
    }
    return q < 0 ? N - 1 : q;
}

// Executed by one full warp.  Returns (to every lane) the smallest fine bin b with
// cum(<= b) >= need, or kFineBins - 1 if the histogram holds fewer than `need` entries;
// *below_out = number of entries in bins < b.  One snapshot of each level is read (all loads in
// flight together).  `top` may lag behind `fine` (fine is incremented first, then a fence, then
// top), never the other way round, so a bound derived from `top` is valid for the true counts.
static __device__ __noinline__ unsigned warp_find_bound(const SelState *st, unsigned need, unsigned *below_out) {
    const unsigned lane = threadIdx.x & 31u;
    // level 1: 2048 coarse bins, 64 per lane
    constexpr int kPerLane = kTopBins / 32;
    unsigned t[kPerLane];
    const unsigned *tp = st->top + lane * kPerLane;
#pragma unroll
    for (int q = 0; q < kPerLane; q += 4) {
        const uint4 v = ld_relaxed_v4(tp + q);
        t[q] = v.x; t[q + 1] = v.y; t[q + 2] = v.z; t[q + 3] = v.w;
    }
    unsigned local = 0;
#pragma unroll
    for (int q = 0; q < kPerLane; ++q) local += t[q];
    unsigned incl = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned u = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += u;
    }
    const unsigned total = __shfl_sync(0xffffffffu, incl, 31);
    if (total < need) {
        if (below_out) *below_out = total;
        return kFineBins - 1u;
    }
    const unsigned cross = __ballot_sync(0xffffffffu, incl >= need);
    const int      owner = __ffs(cross) - 1;
    unsigned c_star = 0, below = 0;
    if ((int)lane == owner) {
        below = incl - local;
        c_star = lane * kPerLane + find_in_lane(t, need, below);
    }
    c_star = __shfl_sync(0xffffffffu, c_star, owner);
    below  = __shfl_sync(0xffffffffu, below, owner);
    // level 2: the 256 fine bins of coarse bin c_star, 8 per lane
    const unsigned *fp = st->fine + (size_t)c_star * 256 + lane * 8;
    const uint4 a = ld_relaxed_v4(fp), b = ld_relaxed_v4(fp + 4);
    const unsigned f[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    unsigned l2 = 0;
#pragma unroll
    for (int q = 0; q < 8; ++q) l2 += f[q];
    unsigned incl2 = l2;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned u = __shfl_up_sync(0xffffffffu, incl2, o);
        if (lane >= o) incl2 += u;
    }
    const unsigned cross2 = __ballot_sync(0xffffffffu, below + incl2 >= need);
    if (cross2 == 0) {                        // cannot happen (fine >= top); no bound rather than a wrong one
        if (below_out) *below_out = below;
        return kFineBins - 1u;
    }
    const int owner2 = __ffs(cross2) - 1;
    unsigned b_star = 0, below2 = 0;
    if ((int)lane == owner2) {
        below2 = below + incl2 - l2;
        b_star = c_star * 256 + lane * 8 + find_in_lane(f, need, below2);
    }
    b_star = __shfl_sync(0xffffffffu, b_star, owner2);
    below2 = __shfl_sync(0xffffffffu, below2, owner2);
    if (below_out) *below_out = below2;
    return b_star;
}

}  // namespace sx

// sx_select.cuh -- selection state shared by the pricing kernels (sx_price.cu) and the top-k
// selection, and the selection itself (select_topk), which runs in topk_select_kernel (sx_topk.cu)
// and inside the fused pricing pass (sx_fused.cu).
//
// While a pricing pass streams the arcs, the violators that can still be among the K most
// violating ones are appended to an unordered candidate list, and a two-level histogram over an
// order-preserving 19-bit image of their reduced cost (sign-stripped exponent + 8 mantissa bits,
// 0.4 % relative width per bin) is kept beside it.  Every `kTightenPeriod` appended candidates the
// appending warp scans the histogram for the smallest bin b* whose cumulative count reaches K and
// lowers `bstar` to it: from then on only violators with bin <= b* are appended (the K-th smallest
// reduced cost lies in a bin <= b*, and counts only grow, so the bound stays valid).  The list
// therefore stays O(K log(n/K)) long however many arcs violate, and the final selection is a
// filter by the final b* plus an all-pairs rank of the few survivors.
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

// ---- the selection of the K <= SX_TOPK_MAX_K best candidates (select_topk) ----------------------
// Executed by every thread of a cooperatively launched grid.  The first kSelThreads threads of a CTA do
// the work; further ones (the fused kernel's TMA producer warp) only join the block barriers.
constexpr int kSelThreads = 256;
constexpr int kDirectCap  = 2048;   // candidate lists up to this length are ranked as they are (the all-pairs
                                    // rank is quadratic: 6990 candidates took 45 us, the filter path 12)
constexpr int kApTile     = 2048;   // elements the rank stages in shared memory at a time
constexpr int kRankCap    = 4096;   // refine until sure + boundary fit this; the rank itself takes up to kSurvCap

// Shared memory of the selection: static in topk_select_kernel, carved out of the TMA stage ring in the
// fused kernel.
struct SelScratch {
    KeyId              tile[kApTile];                  // rank tile
    unsigned           hist[kRefBins];                 // digit histogram of a refinement level
    unsigned long long range[4 * kSelThreads / 32];    // per-warp (key, id) range of a new boundary list
    unsigned           scan[2 * kSelThreads / 32 + 2]; // per-warp list counts + the CTA's list offsets
    unsigned           b[2];                           // bound / digit found by warp 0 and the count below it
};

// The selection's lists at the start of its workspace (sx_topk_workspace_bytes): `sure` (< K elements,
// kSurvCap slots) and two boundary lists of cand_cap elements used by alternate levels.
struct SelLists {
    KeyId *sure, *a, *b;
};
inline SelLists carve_sel_lists(Carver &cv, long long cand_cap) {
    SelLists l;
    l.sure = cv.take<KeyId>(kSurvCap);
    l.a = cv.take<KeyId>(cand_cap > 0 ? cand_cap : 1);
    l.b = cv.take<KeyId>(cand_cap > 0 ? cand_cap : 1);
    return l;
}

// All-pairs rank of n elements given by load(e) (padding sorts last), spread over the grid: L = 1..32 lanes
// share one element and split the comparison range; when the grid has fewer than n * L working threads it
// sweeps the elements in turn.  emit(v, rank, sub, L) is called by the L lanes (sub = 0..L-1) of every real
// element v.
template <class LoadFn, class EmitFn>
__device__ __forceinline__ void all_pairs_rank(int n, LoadFn load, EmitFn emit, KeyId *tile) {
    const int tid = threadIdx.x;
    const int T = gridDim.x * kSelThreads;
    int L = 32;
    while (L > 1 && (long long)n * L > T) L >>= 1;
    const int groups = T / L;                                  // elements ranked per sweep of the grid
    for (int e0 = 0; e0 < n; e0 += groups) {
        const int cta_first = e0 + (blockIdx.x * kSelThreads) / L;
        if (cta_first >= n) break;                             // CTA-uniform
        const int  e = cta_first + tid / L, sub = tid % L;
        const bool active = tid < kSelThreads && e < n;
        KeyId mine{~0ull, 0x7fffffffffffffffll};
        if (active) mine = load(e);
        int cnt = 0;
        for (int t0 = 0; t0 < n; t0 += kApTile) {
            const int tn = n - t0 < kApTile ? n - t0 : kApTile;
            __syncthreads();
            if (tid < kSelThreads)
                for (int j = tid; j < tn; j += kSelThreads) tile[j] = load(t0 + j);
            __syncthreads();
            if (active) {
#pragma unroll 4
                for (int j = sub; j < tn; j += L) cnt += keyid_less(tile[j], mine) ? 1 : 0;
            }
        }
        if (tid < kSelThreads)
            for (int o = L >> 1; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        if (active && mine.key != ~0ull) emit(mine, cnt, sub, L);
    }
}

template <class T> __device__ __forceinline__ T warp_max(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        T w = __shfl_xor_sync(0xffffffffu, v, o);
        v = w > v ? w : v;
    }
    return v;
}

// One partition step of the selection, executed by the whole grid: every element e of this CTA's
// strided share is classified by cls(e) -> 0 (sure), 1 (new boundary list) or 2 (dropped) and
// moved to the end of `sure` / into `bnd`.  Counts are aggregated per CTA (one atomicAdd per list
// and CTA, one set of range atomics per CTA): the classification runs twice, first to count, then
// to scatter.  Also tracks the (key, id) range of the new boundary list for the next level.
template <class LoadFn, class ClsFn>
__device__ __forceinline__ void partition_step(long long n, LoadFn load, ClsFn cls, KeyId *sure, unsigned *n_sure,
                                               KeyId *bnd, unsigned *n_bnd, long long bnd_cap, SelState *st,
                                               int next_level, SelScratch &s) {
    constexpr int kWarps = kSelThreads / 32;
    const bool worker = threadIdx.x < kSelThreads;
    const long long n_mine = worker ? n : 0;                   // elements visible to this thread
    const long long gtid = (long long)blockIdx.x * kSelThreads + threadIdx.x;
    const long long gsz = (long long)gridDim.x * kSelThreads;
    const int lane = lane_id(), warp = threadIdx.x >> 5;
    unsigned c0 = 0, c1 = 0;
    unsigned long long a = 0, b = 0, c = 0, d = 0;      // ~min key, max key, ~min id, max id
    for (long long i = gtid; i < n_mine; i += gsz) {
        const KeyId v = load(i);
        const int k = cls(v);
        c0 += k == 0;
        if (k == 1) {
            ++c1;
            const unsigned long long id = (unsigned long long)v.id;
            a = ~v.key > a ? ~v.key : a; b = v.key > b ? v.key : b;
            c = ~id > c ? ~id : c;       d = id > d ? id : d;
        }
    }
    // block-exclusive scan of (c0, c1)
    unsigned i0 = c0, i1 = c1;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned t0 = __shfl_up_sync(0xffffffffu, i0, o), t1 = __shfl_up_sync(0xffffffffu, i1, o);
        if (lane >= o) { i0 += t0; i1 += t1; }
    }
    a = warp_max(a); b = warp_max(b); c = warp_max(c); d = warp_max(d);
    __syncthreads();
    if (worker && lane == 31) { s.scan[warp] = i0; s.scan[kWarps + warp] = i1; }
    if (worker && lane == 0) { s.range[warp * 4] = a; s.range[warp * 4 + 1] = b; s.range[warp * 4 + 2] = c; s.range[warp * 4 + 3] = d; }
    __syncthreads();
    if (threadIdx.x >= 32 && threadIdx.x < 36) {        // one range atomic per CTA and quantity
        const int q = threadIdx.x - 32;
        unsigned long long m = 0;
        for (int w = 0; w < kWarps; ++w) m = s.range[w * 4 + q] > m ? s.range[w * 4 + q] : m;
        unsigned long long *dst = q == 0 ? st->inv_kmin : (q == 1 ? st->kmax : (q == 2 ? st->inv_imin : st->imax));
        if (m) atomicMax(&dst[next_level], m);
    }
    if (threadIdx.x == 0) {
        unsigned t0 = 0, t1 = 0;
        for (int w = 0; w < kWarps; ++w) {
            const unsigned x0 = s.scan[w], x1 = s.scan[kWarps + w];
            s.scan[w] = t0; s.scan[kWarps + w] = t1;
            t0 += x0; t1 += x1;
        }
        s.scan[2 * kWarps] = t0 ? atomicAdd(n_sure, t0) : 0u;
        s.scan[2 * kWarps + 1] = t1 ? atomicAdd(n_bnd, t1) : 0u;
    }
    __syncthreads();
    if (!worker) return;
    unsigned p0 = s.scan[2 * kWarps] + s.scan[warp] + i0 - c0;
    unsigned p1 = s.scan[2 * kWarps + 1] + s.scan[kWarps + warp] + i1 - c1;
    for (long long i = gtid; i < n; i += gsz) {
        const KeyId v = load(i);
        const int k = cls(v);
        if (k == 0) { if (p0 < (unsigned)kSurvCap) sure[p0] = v; ++p0; }
        else if (k == 1) { if ((long long)p1 < bnd_cap) bnd[p1] = v; ++p1; }
    }
}

// Refinement levels of select_topk, after level 0 left `sure` and the boundary list `a` (level 0 of the
// state).  While sure + boundary > kRankCap: an 11-bit digit of (key, id) taken at the highest bit in which
// the boundary list's minimum and maximum differ is histogrammed, the digit d* that holds the remaining
// rank `need` is found, digits < d* become sure, == d* the new boundary list (in `b`, then `a` again, ...).
// Near-ties resolve in one level, exact ties fall through to the id.  Returns the level of the final
// boundary list, or -1 when only copies of one (key, id) pair are left and they do not fit kSurvCap.
// Not inlined: the fused kernel's pricing loop keeps its register allocation.
template <class GridSync>
__device__ __noinline__ int refine_boundary(SelState *st, long long need, SelLists l, long long cap, SelScratch &s,
                                            GridSync grid_sync) {
    // Each level leaves a list that agrees on every bit from the chosen digit's lowest bit up, so 6 levels
    // settle the 64-bit key and 6 more the 63-bit id: only copies of one (key, id) can reach kMaxLevels.
    static_assert(kMaxLevels >= (64 + 10) / 11 + (63 + 10) / 11, "refinement levels cannot settle a (key, id)");
    const bool worker = threadIdx.x < kSelThreads;
    const long long gtid = (long long)blockIdx.x * kSelThreads + threadIdx.x;
    const long long gsz = (long long)gridDim.x * kSelThreads;
    KeyId *listA = l.a, *listB = l.b;
    for (int level = 0;; ++level) {
        const unsigned n_sure = ld_relaxed_u32(&st->n_sure), n_a = ld_relaxed_u32(&st->n_list[level]);
        if (n_sure + n_a <= (unsigned)kRankCap) return level;
        if (level == kMaxLevels) return n_sure + n_a > (unsigned)kSurvCap ? -1 : level;
        const unsigned long long kmin = ~__ldcg(&st->inv_kmin[level]), kmax = __ldcg(&st->kmax[level]);
        const unsigned long long imin = ~__ldcg(&st->inv_imin[level]), imax = __ldcg(&st->imax[level]);
        const bool by_key = kmin != kmax;
        const unsigned long long diff = by_key ? (kmin ^ kmax) : (imin ^ imax);
        if (diff == 0) return n_sure + n_a > (unsigned)kSurvCap ? -1 : level;   // duplicates of one (key, id)
        const int p = 63 - __clzll((long long)diff);
        const int sh = p > 10 ? p - 10 : 0;
        auto digit = [&](const KeyId &v) {
            return (unsigned)(((by_key ? v.key : (unsigned long long)v.id) >> sh) & (kRefBins - 1));
        };
        if (worker)
            for (int i = threadIdx.x; i < kRefBins; i += kSelThreads) s.hist[i] = 0;
        __syncthreads();
        if (worker) {   // digit histogram; lanes holding the same digit add once (near-ties share one digit)
            const long long na_ceil = ((long long)n_a + 31) / 32 * 32;
            for (long long i = gtid; i < na_ceil; i += gsz) {
                const unsigned dg = i < n_a ? digit(ld_keyid(listA + i)) : 0xffffffffu;
                const unsigned peers = __match_any_sync(0xffffffffu, dg);
                if (dg != 0xffffffffu && (int)lane_id() == __ffs(peers) - 1) atomicAdd(&s.hist[dg], (unsigned)__popc(peers));
            }
        }
        __syncthreads();
        if (worker)
            for (int i = threadIdx.x; i < kRefBins; i += kSelThreads)
                if (s.hist[i]) atomicAdd(&st->hist2[level][i], s.hist[i]);
        grid_sync();
        // digit holding rank `need`: 2048 bins, 64 per lane of warp 0
        if (threadIdx.x < 32) {
            const unsigned *h = st->hist2[level] + threadIdx.x * 64;
            unsigned hv[64];
#pragma unroll
            for (int q = 0; q < 64; q += 4) {
                const uint4 v = __ldcg(reinterpret_cast<const uint4 *>(h + q));
                hv[q] = v.x; hv[q + 1] = v.y; hv[q + 2] = v.z; hv[q + 3] = v.w;
            }
            unsigned local = 0;
#pragma unroll
            for (int q = 0; q < 64; ++q) local += hv[q];
            unsigned incl = local;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
                if (threadIdx.x >= o) incl += t;
            }
            const unsigned cross = __ballot_sync(0xffffffffu, (long long)incl >= need);
            const int owner = cross ? __ffs(cross) - 1 : 31;
            if ((int)threadIdx.x == owner) {
                unsigned cum = incl - local;
                const int q = find_in_lane(hv, (unsigned)need, cum);
                s.b[0] = threadIdx.x * 64 + q;
                s.b[1] = cum;
            }
        }
        __syncthreads();
        const unsigned dstar = s.b[0];
        need -= (long long)s.b[1];
        partition_step(
            (long long)n_a, [&](long long i) { return ld_keyid(listA + i); },
            [&](const KeyId &v) {
                const unsigned dg = digit(v);
                return dg < dstar ? 0 : (dg == dstar ? 1 : 2);
            },
            l.sure, &st->n_sure, listB, &st->n_list[level + 1], cap, st, level + 1, s);
        grid_sync();
        KeyId *t = listA; listA = listB; listB = t;
    }
}

struct SelResult {
    int  n_out;        // min(elements ranked, K): output positions 0 .. n_out - 1 are emitted
    bool duplicates;   // only copies of one (rc, id) pair were left: nothing is emitted (SX_STATUS_DUPLICATE_CANDIDATES)
};

// The K smallest by (rc, id) of the n candidates (cand_rc, cand_id), in one cooperative launch; written by
// other CTAs of the same kernel or by an earlier one (the candidates are read through L2).  `st` is the
// state the pricing pass filled: its histogram gives the level-0 bound, its scratch fields start at zero.
// grid_sync() is the grid-wide barrier; emit(v, rank, sub, L) as in all_pairs_rank (rank can be >= K).
//   direct    a list of at most kDirectCap candidates is ranked as it is;
//   level 0   otherwise the candidates are split by the pricing histogram's final bound b*: bin < b* are
//             "sure" (there are fewer than K of them), bin == b* form the boundary list, the rest is dropped;
//   refine    refine_boundary, while sure + boundary > kRankCap;
//   rank      all-pairs rank of sure ++ boundary (<= kSurvCap elements) gives every output position.
template <class GridSync, class EmitFn>
__device__ __forceinline__ SelResult select_topk(const double *cand_rc, const long long *cand_id, long long n,
                                                 long long cap, SelState *st, int K, SelLists l, SelScratch &s,
                                                 GridSync grid_sync, EmitFn emit) {
    auto cand = [&](long long i) { return KeyId{f64_to_sort_key(__ldcg(cand_rc + i)), __ldcg(cand_id + i)}; };
    if (n <= kDirectCap) {
        all_pairs_rank((int)n, cand, emit, s.tile);
        return SelResult{n < K ? (int)n : K, false};
    }
    // ---- level 0: split by the pricing histogram ----
    if (threadIdx.x < 32) {
        unsigned below = 0;
        const unsigned b = warp_find_bound(st, (unsigned)K, &below);
        if (threadIdx.x == 0) { s.b[0] = b; s.b[1] = below; }
    }
    __syncthreads();
    const unsigned b1 = s.b[0];
    const long long need = (long long)K - (long long)s.b[1];     // rank still to find inside the boundary list
    partition_step(
        n, cand,
        [&](const KeyId &v) {
            const unsigned long long kb = v.key >> (64 - 1 - kFineBits);                 // = cand_bin(rc)
            const unsigned bin = kb < (unsigned long long)kFineBins ? (unsigned)kb : kFineBins - 1u;
            return bin < b1 ? 0 : (bin == b1 ? 1 : 2);
        },
        l.sure, &st->n_sure, l.a, &st->n_list[0], cap, st, 0, s);
    grid_sync();
    const int level = refine_boundary(st, need, l, cap, s, grid_sync);
    if (level < 0) return SelResult{0, true};
    // ---- all-pairs rank of sure ++ boundary ----
    const KeyId *bnd = (level & 1) ? l.b : l.a;
    const int n_sure = (int)ld_relaxed_u32(&st->n_sure);
    const int n_s = n_sure + (int)ld_relaxed_u32(&st->n_list[level]);
    all_pairs_rank(n_s, [&](int e) { return ld_keyid(e < n_sure ? l.sure + e : bnd + (e - n_sure)); }, emit, s.tile);
    return SelResult{n_s < K ? n_s : K, false};
}

}  // namespace sx

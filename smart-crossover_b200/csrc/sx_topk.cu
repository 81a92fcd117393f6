// sx_topk.cu -- selection of the K most violating arcs (sm_100a).
//
// north_star extension (SURVEY.md section 8 row a9; the reference never ranks violators, it
// only tests `np.all(rc >= -tol)`, net_manager.py:318,496): among the candidates (rc, arc id)
// compacted by the pricing kernels, return the K smallest by (rc ascending, id ascending).
// (rc, id) is a strict total order, so the result does not depend on the (unordered)
// compaction or on how many GPUs priced the matrix.
//
// K <= 1024: ONE cooperative launch (topk_select_kernel), no host round trip:
//   1. filter: the pricing kernels left a histogram of the candidates' reduced costs
//      (sx_select.cuh); b* = the smallest bin whose cumulative count reaches K.  Candidates
//      with bin < b* are among the K best, bin b* (0.4 % wide) is the boundary list;
//   2. refine: while the list is too long, an 11-bit digit of (key, id) splits the boundary list
//      again; a list of distinct (key, id) pairs shrinks to one element within 12 levels;
//   3. all-pairs rank: every survivor counts the survivors below it; that count is its
//      position in the output.  O(n_surv^2) compares spread over the whole GPU (1 to 32 lanes
//      per element), a few microseconds for the typical 1-2 K survivors.
//   The candidates must be distinct arcs.  Only copies of one (rc, id) pair -- the same arc priced
//   into one pass many times -- can keep the list long; the selection is then void and raises
//   SX_STATUS_DUPLICATE_CANDIDATES in the pricing header.
// K > 1024: two stable radix argsorts (by id, then by rc) over the candidates.
// Merge of G sorted, padded per-GPU lists after the exchange (sx_topk_merge): an element's position is
// the number of entries below it in every list (binary searches).
#include <math.h>

#include <cooperative_groups.h>

#include "sx_common.cuh"
#include "sx_select.cuh"
#include "sx_ll.cuh"

namespace cg = cooperative_groups;

namespace sx {

struct Cand {
    double    rc;
    long long id;
};
__device__ __forceinline__ Cand cand_pad() { return Cand{INFINITY, -1}; }
// padding must sort after every real candidate: compare as (+inf, max id)
__device__ __forceinline__ bool cand_less_p(const Cand &a, const Cand &b) {
    const long long ia = a.id < 0 ? 0x7fffffffffffffffll : a.id;
    const long long ib = b.id < 0 ? 0x7fffffffffffffffll : b.id;
    return a.rc < b.rc || (a.rc == b.rc && ia < ib);
}

__device__ __forceinline__ Cand shfl_xor_cand(const Cand &c, int mask) {
    Cand r;
    r.rc = __shfl_xor_sync(0xffffffffu, c.rc, mask);
    r.id = __shfl_xor_sync(0xffffffffu, c.id, mask);
    return r;
}

// number of elements of a sorted, padded list prefix [0, len) that are  < x  (strict)
__device__ __forceinline__ int lower_bound_list(const double *rc, const long long *id, int len, const Cand &x) {
    int lo = 0, hi = len;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const Cand m{rc[mid], id[mid]};
        if (cand_less_p(m, x)) lo = mid + 1; else hi = mid;
    }
    return lo;
}
// number of elements <= x
__device__ __forceinline__ int upper_bound_list(const double *rc, const long long *id, int len, const Cand &x) {
    int lo = 0, hi = len;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const Cand m{rc[mid], id[mid]};
        if (!cand_less_p(x, m)) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// Rank merge of sx_topk_merge when G * K > 2^22 (too many elements for one thread each), step 1 (one CTA).
// lists: L sorted, padded lists of length K.
//   thr      = smallest last element over the lists: the global K-th best is <= it, so only the
//              prefix of each list with elements <= thr can be in the answer;
//   plen[l]  = length of that prefix;  poff[l] = exclusive prefix sum;  poff[L] = work total.
__global__ void __launch_bounds__(1024)
topk_prep_kernel(const double *__restrict__ lists_rc, const long long *__restrict__ lists_id, long long LS, int L,
                 int K, int *__restrict__ plen, int *__restrict__ poff, double *__restrict__ out_rc, long long *__restrict__ out_id,
                 long long *out_n, const long long *headers, long long *out_summary) {
    // outputs start as padding; the rank kernel (next launch) overwrites the first out_n entries
    for (int i = threadIdx.x; i < K; i += blockDim.x) { out_rc[i] = INFINITY; out_id[i] = -1; }
    if (headers && out_summary && threadIdx.x == 0) {
        // fold the per-rank pricing headers {n_violating, min_rc_key}: total, min, largest single count
        long long tot = 0, mn = 0x7fffffffffffffffll, mx = 0, stt = 0;
        for (int l = 0; l < L; ++l) {
            const long long c = headers[(long long)l * LS], k = headers[(long long)l * LS + 1];
            tot += c; mn = k < mn ? k : mn; mx = c > mx ? c : mx; stt |= headers[(long long)l * LS + 3];
        }
        out_summary[0] = tot; out_summary[1] = mn; out_summary[2] = mx; out_summary[3] = stt;
    }
    __shared__ Cand s_thr[32];
    __shared__ int  s_warp[32];
    __shared__ int  s_carry;
    const int lane = lane_id(), warp = threadIdx.x >> 5;
    __shared__ long long s_red[32];
    auto block_sum = [&](long long v) -> long long {
        v = warp_sum(v);
        __syncthreads();
        if (lane == 0) s_red[warp] = v;
        __syncthreads();
        long long t = 0;
        for (int w = 0; w < 32; ++w) t += s_red[w];
        return t;
    };
    auto block_min_cand = [&](Cand c, bool want_max) -> Cand {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const Cand other = shfl_xor_cand(c, o);
            if (cand_less_p(other, c) != want_max) c = other;
        }
        __syncthreads();
        if (lane == 0) s_thr[warp] = c;
        __syncthreads();
        Cand r = s_thr[0];
        for (int w = 1; w < 32; ++w) if (cand_less_p(s_thr[w], r) != want_max) r = s_thr[w];
        return r;
    };
    if (threadIdx.x == 0) s_carry = 0;
    // bound 1: the smallest "last element of a list" (padding = +inf: no constraint)
    Cand thr = cand_pad();
    long long n_real_lists = 0;
    for (int l = threadIdx.x; l < L; l += blockDim.x) {
        const long long *ids = lists_id + (long long)l * LS;
        const Cand c{lists_rc[(long long)l * LS + K - 1], ids[K - 1]};
        if (cand_less_p(c, thr)) thr = c;
        int lo = 0, hi = K;                              // real length of the list: first padding entry
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (ids[mid] >= 0) lo = mid + 1; else hi = mid; }
        plen[l] = lo;
        n_real_lists += lo;
    }
    thr = block_min_cand(thr, false);
    // bound 2: the smallest depth i with sum_l min(len_l, i) >= K; the union of the depth-i prefixes
    // already holds K elements, so the global K-th best is <= the largest element among them.  Much
    // tighter than bound 1 when there are many lists.
    const long long all_real = block_sum(n_real_lists);
    if (all_real >= K) {
        int lo = 1, hi = K;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            long long part = 0;
            for (int l = threadIdx.x; l < L; l += blockDim.x) part += plen[l] < mid ? plen[l] : mid;
            if (block_sum(part) >= K) hi = mid; else lo = mid + 1;
        }
        Cand deep = Cand{-INFINITY, 0};
        for (int l = threadIdx.x; l < L; l += blockDim.x) {
            const int take = plen[l] < lo ? plen[l] : lo;
            if (take > 0) {
                const Cand c{lists_rc[(long long)l * LS + take - 1], lists_id[(long long)l * LS + take - 1]};
                if (cand_less_p(deep, c)) deep = c;
            }
        }
        deep = block_min_cand(deep, true);
        if (cand_less_p(deep, thr)) thr = deep;
    }
    __syncthreads();
    // prefix lengths and their exclusive scan, 1024 lists per sweep
    long long real_total = 0;
    for (int base = 0; base < L; base += blockDim.x) {
        const int l = base + threadIdx.x;
        int len = 0;
        if (l < L) len = upper_bound_list(lists_rc + (long long)l * LS, lists_id + (long long)l * LS, K, thr);
        // do not count padding (id < 0) that ties with an all-padding threshold
        if (l < L && len > 0) {
            int lo = 0, hi = len;                       // first padding entry within [0, len)
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (lists_id[(long long)l * LS + mid] >= 0) lo = mid + 1; else hi = mid; }
            len = lo;
        }
        int incl = len;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        int add = s_carry;
        for (int w = 0; w < warp; ++w) add += s_warp[w];
        if (l < L) { plen[l] = len; poff[l] = add + incl - len; }
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) s_carry = add + incl;
        __syncthreads();
        real_total = s_carry;
    }
    if (threadIdx.x == 0) {
        poff[L] = (int)real_total;
        *out_n = real_total < K ? real_total : K;
    }
}

// Rank merge, step 2: one WARP per surviving element; lanes split the lists, each does a binary
// search in that list's prefix, a shuffle reduction gives the global rank.
__global__ void __launch_bounds__(256)
topk_rank_kernel(const double *__restrict__ lists_rc, const long long *__restrict__ lists_id, long long LS, int L,
                 int K, const int *__restrict__ plen, const int *__restrict__ poff,
                 double *__restrict__ out_rc, long long *__restrict__ out_id) {
    const int lane = lane_id();
    const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
    const int total = poff[L];
    for (long long w = (((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5); w < total; w += n_warps) {
        // list owning work item w: last l with poff[l] <= w
        int lo = 0, hi = L;
        while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (poff[mid] <= w) lo = mid; else hi = mid; }
        const int l = lo, i = (int)(w - poff[l]);
        const Cand c{lists_rc[(long long)l * LS + i], lists_id[(long long)l * LS + i]};
        int rank = 0;
        for (int m = lane; m < L; m += 32) {
            if (m == l) rank += i;
            else {
                const int len = plen[m];
                if (len) rank += lower_bound_list(lists_rc + (long long)m * LS, lists_id + (long long)m * LS, len, c);
            }
        }
        rank = warp_sum(rank);
        if (lane == 0 && rank < K) { out_rc[rank] = c.rc; out_id[rank] = c.id; }
    }
}

// ---- fast path ----------------------------------------------------------------------------
constexpr int kApThreads = 256;
constexpr int kApTile    = 2048;
constexpr int kRankCap   = 4096;   // refine until sure + boundary fit this; the rank itself takes up to kSurvCap

// All-pairs rank of n elements given by load(e) (padding sorts last).  Every thread of the grid
// takes part; L = 1..32 lanes share one element and split the comparison range.  emit(e, rank)
// is called once per real element.  Needs n <= gridDim.x * kApThreads.
template <class LoadFn, class EmitFn>
__device__ __forceinline__ void all_pairs_rank(int n, LoadFn load, EmitFn emit) {
    __shared__ KeyId tile[kApTile];
    const int T = gridDim.x * kApThreads;
    int L = 32;
    while (L > 1 && (long long)n * L > T) L >>= 1;
    const int gtid = blockIdx.x * kApThreads + threadIdx.x;
    const int e = gtid / L, sub = gtid % L;
    if ((blockIdx.x * kApThreads) / L >= n) return;            // CTA-uniform: nothing to rank here
    KeyId mine{~0ull, 0x7fffffffffffffffll};
    const bool real = e < n;
    if (real) mine = load(e);
    const bool valid = real && mine.key != ~0ull;
    int cnt = 0;
    for (int t0 = 0; t0 < n; t0 += kApTile) {
        const int tn = n - t0 < kApTile ? n - t0 : kApTile;
        __syncthreads();
        for (int j = threadIdx.x; j < tn; j += kApThreads) tile[j] = load(t0 + j);
        __syncthreads();
        if (valid) {
#pragma unroll 4
            for (int j = sub; j < tn; j += L) cnt += keyid_less(tile[j], mine) ? 1 : 0;
        }
    }
    for (int o = L >> 1; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (valid && sub == 0) emit(e, cnt);
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
                                               int next_level, unsigned *s_scan /* 2 * 8 + 2 words */,
                                               unsigned long long *s_range /* 8 * 4 */) {
    const long long gtid = (long long)blockIdx.x * kApThreads + threadIdx.x;
    const long long gsz = (long long)gridDim.x * kApThreads;
    const int lane = lane_id(), warp = threadIdx.x >> 5;
    unsigned c0 = 0, c1 = 0;
    unsigned long long a = 0, b = 0, c = 0, d = 0;      // ~min key, max key, ~min id, max id
    for (long long i = gtid; i < n; i += gsz) {
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
    if (lane == 31) { s_scan[warp] = i0; s_scan[8 + warp] = i1; }
    if (lane == 0) { s_range[warp * 4] = a; s_range[warp * 4 + 1] = b; s_range[warp * 4 + 2] = c; s_range[warp * 4 + 3] = d; }
    __syncthreads();
    if (threadIdx.x >= 32 && threadIdx.x < 36) {        // one range atomic per CTA and quantity
        const int q = threadIdx.x - 32;
        unsigned long long m = 0;
        for (int w = 0; w < kApThreads / 32; ++w) m = s_range[w * 4 + q] > m ? s_range[w * 4 + q] : m;
        unsigned long long *dst = q == 0 ? st->inv_kmin : (q == 1 ? st->kmax : (q == 2 ? st->inv_imin : st->imax));
        if (m) atomicMax(&dst[next_level], m);
    }
    if (threadIdx.x == 0) {
        unsigned t0 = 0, t1 = 0;
        for (int w = 0; w < kApThreads / 32; ++w) {
            const unsigned x0 = s_scan[w], x1 = s_scan[8 + w];
            s_scan[w] = t0; s_scan[8 + w] = t1;
            t0 += x0; t1 += x1;
        }
        s_scan[16] = t0 ? atomicAdd(n_sure, t0) : 0u;
        s_scan[17] = t1 ? atomicAdd(n_bnd, t1) : 0u;
    }
    __syncthreads();
    unsigned p0 = s_scan[16] + s_scan[warp] + i0 - c0;
    unsigned p1 = s_scan[17] + s_scan[8 + warp] + i1 - c1;
    for (long long i = gtid; i < n; i += gsz) {
        const KeyId v = load(i);
        const int k = cls(v);
        if (k == 0) { if (p0 < (unsigned)kSurvCap) sure[p0] = v; ++p0; }
        else if (k == 1) { if ((long long)p1 < bnd_cap) bnd[p1] = v; ++p1; }
    }
}

// The whole selection in ONE cooperative launch (K <= 1024):
//   level 0   candidates are split by the pricing histogram's final bound b*: bin < b* are "sure"
//             (there are fewer than K of them), bin == b* form the boundary list, the rest is dropped;
//   refine    while sure + boundary > kSurvCap: an 11-bit digit of (key, id) taken at the highest bit
//             in which the boundary list's minimum and maximum differ is histogrammed, the digit d*
//             that holds the remaining rank is found, digits < d* become sure, == d* the new boundary
//             list.  Near-ties resolve in one level, exact ties fall through to the id;
//   rank      all-pairs rank of sure + boundary (<= 8192 elements) gives every output position.
__global__ void __launch_bounds__(kApThreads)
topk_select_kernel(const double *__restrict__ cand_rc, const long long *__restrict__ cand_id, long long cand_cap,
                   SelState *st, sx_price_header *hdr, int K, KeyId *sure, KeyId *listA, KeyId *listB,
                   double *__restrict__ out_rc, long long *__restrict__ out_id, long long *out_n) {
    cg::grid_group grid = cg::this_grid();
    __shared__ unsigned s_hist[kRefBins];
    __shared__ unsigned s_b[2];
    __shared__ unsigned s_scan[18];
    __shared__ unsigned long long s_range[32];
    const unsigned long long n64 = st->n_cand;
    long long n = (long long)n64;
    if (n64 > (unsigned long long)cand_cap) {
        n = cand_cap;
        if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(&hdr->status, kStatusCandOverflow);
    }
    // the candidate list was pruned for the K given to sx_price_pass_begin: a larger K here cannot be served
    if ((unsigned)K > st->K && blockIdx.x == 0 && threadIdx.x == 0) atomicOr(&hdr->status, kStatusKMismatch);
    const long long gtid = (long long)blockIdx.x * kApThreads + threadIdx.x;
    const long long gsz = (long long)gridDim.x * kApThreads;

    // ---- level 0: split by the pricing histogram ----
    if (threadIdx.x < 32) {
        unsigned below = 0;
        const unsigned b = warp_find_bound(st, (unsigned)K, &below);
        if (threadIdx.x == 0) { s_b[0] = b; s_b[1] = below; }
    }
    __syncthreads();
    const unsigned b1 = s_b[0];
    long long need = (long long)K - (long long)s_b[1];          // rank still to find inside the boundary list
    partition_step(
        n, [&](long long i) { return KeyId{f64_to_sort_key(cand_rc[i]), cand_id[i]}; },
        [&](const KeyId &v) {
            const unsigned long long kb = v.key >> (64 - 1 - kFineBits);                 // = cand_bin(rc)
            const unsigned bin = kb < (unsigned long long)kFineBins ? (unsigned)kb : kFineBins - 1u;
            return bin < b1 ? 0 : (bin == b1 ? 1 : 2);
        },
        sure, &st->n_sure, listA, &st->n_list[0], cand_cap, st, 0, s_scan, s_range);
    grid.sync();

    // ---- refinement levels ----
    // Each level leaves a list that agrees on every bit from the chosen digit's lowest bit up, so 6 levels
    // settle the 64-bit key and 6 more the 63-bit id: only copies of one (key, id) can reach kMaxLevels.
    static_assert(kMaxLevels >= (64 + 10) / 11 + (63 + 10) / 11, "refinement levels cannot settle a (key, id)");
    int level = 0;
    bool failed = false;
    for (;; ++level) {
        const unsigned n_sure = ld_relaxed_u32(&st->n_sure), n_a = ld_relaxed_u32(&st->n_list[level]);
        if (n_sure + n_a <= (unsigned)kRankCap) break;
        if (level == kMaxLevels) { failed = n_sure + n_a > (unsigned)kSurvCap; break; }
        const unsigned long long kmin = ~__ldcg(&st->inv_kmin[level]), kmax = __ldcg(&st->kmax[level]);
        const unsigned long long imin = ~__ldcg(&st->inv_imin[level]), imax = __ldcg(&st->imax[level]);
        const bool by_key = kmin != kmax;
        const unsigned long long diff = by_key ? (kmin ^ kmax) : (imin ^ imax);
        if (diff == 0) { failed = n_sure + n_a > (unsigned)kSurvCap; break; }   // duplicates of one (key, id)
        const int p = 63 - __clzll((long long)diff);
        const int sh = p > 10 ? p - 10 : 0;
        auto digit = [&](const KeyId &v) {
            return (unsigned)(((by_key ? v.key : (unsigned long long)v.id) >> sh) & (kRefBins - 1));
        };
        for (int i = threadIdx.x; i < kRefBins; i += kApThreads) s_hist[i] = 0;
        __syncthreads();
        {   // digit histogram; lanes holding the same digit add once (near-ties share one digit)
            const long long na_ceil = ((long long)n_a + 31) / 32 * 32;
            for (long long i = gtid; i < na_ceil; i += gsz) {
                const unsigned dg = i < n_a ? digit(ld_keyid(listA + i)) : 0xffffffffu;
                const unsigned peers = __match_any_sync(0xffffffffu, dg);
                if (dg != 0xffffffffu && (int)lane_id() == __ffs(peers) - 1) atomicAdd(&s_hist[dg], (unsigned)__popc(peers));
            }
        }
        __syncthreads();
        for (int i = threadIdx.x; i < kRefBins; i += kApThreads)
            if (s_hist[i]) atomicAdd(&st->hist2[level][i], s_hist[i]);
        grid.sync();
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
                s_b[0] = threadIdx.x * 64 + q;
                s_b[1] = cum;
            }
        }
        __syncthreads();
        const unsigned dstar = s_b[0];
        need -= (long long)s_b[1];
        partition_step(
            (long long)n_a, [&](long long i) { return ld_keyid(listA + i); },
            [&](const KeyId &v) {
                const unsigned dg = digit(v);
                return dg < dstar ? 0 : (dg == dstar ? 1 : 2);
            },
            sure, &st->n_sure, listB, &st->n_list[level + 1], cand_cap, st, level + 1, s_scan, s_range);
        grid.sync();
        KeyId *t = listA; listA = listB; listB = t;
    }

    // ---- all-pairs rank of sure ++ boundary ----
    const int n_sure = failed ? 0 : (int)ld_relaxed_u32(&st->n_sure);
    const int n_s = failed ? 0 : n_sure + (int)ld_relaxed_u32(&st->n_list[level]);
    const int n_out = n_s < K ? n_s : K;
    if (blockIdx.x == 0) {
        for (int i = n_out + threadIdx.x; i < K; i += kApThreads) { out_rc[i] = INFINITY; out_id[i] = -1; }
        if (threadIdx.x == 0) {
            *out_n = n_out;
            if (failed) atomicOr(&hdr->status, kStatusDuplicateCandidates);
        }
    }
    if (n_s == 0) return;
    all_pairs_rank(
        n_s, [&](int e) { return ld_keyid(e < n_sure ? sure + e : listA + (e - n_sure)); },
        [&](int e, int rank) {
            if (rank < K) {
                const KeyId v = ld_keyid(e < n_sure ? sure + e : listA + (e - n_sure));
                out_rc[rank] = sort_key_to_f64(v.key);
                out_id[rank] = v.id;
            }
        });
}

// Merge of G sorted, padded blocks of K (exchanged between G ranks).  One thread per element: its
// position in the merged order is its index in its own block plus, for every other block, the number
// of entries below it (binary search; (rc, id) is a strict total order and ids are distinct across
// blocks).  G * 10 dependent L1/L2 loads per element instead of an all-pairs pass over G * K.
__device__ __forceinline__ KeyId merge_load(const double *rc, const long long *id, long long off) {
    const long long i = id[off];
    return i < 0 ? KeyId{~0ull, 0x7fffffffffffffffll} : KeyId{f64_to_sort_key(rc[off]), i};
}

__global__ void __launch_bounds__(1024)
merge_rank_kernel(const double *blocks_rc, const long long *blocks_id, long long LS, int G,
                  int K, const long long *headers, double *__restrict__ out_rc, long long *__restrict__ out_id,
                  long long *out_n, long long *out_summary, const unsigned long long *parity_ctr,
                  long long parity_stride, int use_smem) {
    if (parity_ctr) {   // double-buffered exchange: the blocks of this epoch are in half (epoch & 1)
        const long long off = (long long)(*parity_ctr & 1ull) * parity_stride;
        blocks_rc += off; blocks_id += off;
        if (headers) headers += off;
    }
    const int n = G * K;
    // Stage every block's (key, id) in shared memory when it fits (coalesced loads, then ~G * 10 shared
    // loads per element); otherwise search the blocks in global memory.
    extern __shared__ __align__(16) unsigned char mg_raw[];
    KeyId *stage = reinterpret_cast<KeyId *>(mg_raw);
    __shared__ int s_real;
    __shared__ long long s_hdr[4];
    if (threadIdx.x == 0) { s_real = 0; s_hdr[0] = 0; s_hdr[1] = 0x7fffffffffffffffll; s_hdr[2] = 0; s_hdr[3] = 0; }
    __syncthreads();
    int my_real = 0;
    if (use_smem) {
        for (int e = threadIdx.x; e < n; e += blockDim.x) {
            const int g = e / K;
            const KeyId v = merge_load(blocks_rc, blocks_id, (long long)g * LS + (e - g * K));
            stage[e] = v;
            my_real += v.key != ~0ull;
        }
    }
    if (blockIdx.x == 0) {
        if (!use_smem) {
            // real entries per block = first padding slot (ids are -1 from there on)
            for (int g = threadIdx.x; g < G; g += blockDim.x) {
                int lo = 0, hi = K;
                while (lo < hi) { const int mid = (lo + hi) >> 1; if (blocks_id[(long long)g * LS + mid] >= 0) lo = mid + 1; else hi = mid; }
                my_real += lo;
            }
        }
        my_real = warp_sum(my_real);
        if (lane_id() == 0 && my_real) atomicAdd(&s_real, my_real);
        if (headers && out_summary) {
            // fold the per-rank pricing headers: total count, min key, largest single count, status bits
            for (int g = threadIdx.x; g < G; g += blockDim.x) {
                const long long *h = headers + (long long)g * LS;
                atomicAdd((unsigned long long *)&s_hdr[0], (unsigned long long)h[0]);
                atomicMin(&s_hdr[1], h[1]);
                atomicMax(&s_hdr[2], h[0]);
                atomicOr((unsigned long long *)&s_hdr[3], (unsigned long long)h[3]);
            }
        }
    }
    __syncthreads();
    if (blockIdx.x == 0) {
        const int n_out = s_real < K ? s_real : K;             // outputs past the total are padding
        for (int i = n_out + threadIdx.x; i < K; i += blockDim.x) { out_rc[i] = INFINITY; out_id[i] = -1; }
        if (threadIdx.x == 0) {
            *out_n = n_out;
            if (headers && out_summary) {
                out_summary[0] = s_hdr[0]; out_summary[1] = s_hdr[1]; out_summary[2] = s_hdr[2]; out_summary[3] = s_hdr[3];
            }
        }
    }
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
        const int g = e / K, i = e - g * K;
        const KeyId mine = use_smem ? stage[e] : merge_load(blocks_rc, blocks_id, (long long)g * LS + i);
        if (mine.key == ~0ull) continue;                       // padding
        int rank = i;
        for (int h = 0; h < G && rank < K; ++h) {
            if (h == g) continue;
            const long long base = (long long)h * LS;
            int lo = 0, hi = K;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                const KeyId other = use_smem ? stage[h * K + mid] : merge_load(blocks_rc, blocks_id, base + mid);
                if (keyid_less(other, mine)) lo = mid + 1; else hi = mid;
            }
            rank += lo;
        }
        if (rank < K) { out_rc[rank] = blocks_rc[(long long)g * LS + i]; out_id[rank] = mine.id; }
    }
}

// Merge straight out of the LL exchange buffer (sx_exchange_push_ll): staging a block in shared memory
// IS the wait for it -- every slot is polled until both of its flags show this epoch.
__global__ void __launch_bounds__(1024)
merge_ll_kernel(char *ll_buf, long long block_len, int G, int K, double *__restrict__ out_rc,
                long long *__restrict__ out_id, long long *out_n, long long *out_summary, int *status,
                unsigned long long timeout_ns) {
    extern __shared__ __align__(16) unsigned char mg_raw[];
    KeyId *stage = reinterpret_cast<KeyId *>(mg_raw);
    __shared__ int s_real;
    __shared__ long long s_hdr[4];
    const size_t slots_bytes = (size_t)2 * G * block_len * 16;
    // The merge keeps an epoch counter of its own ([2], [3] = CTAs done), advanced once per launch like the
    // pushing side's ([0], [1]): it depends on no other kernel of this GPU, so it may be launched with
    // programmatic stream serialisation and become resident while the pricing kernel is still draining.
    unsigned long long *mctr = reinterpret_cast<unsigned long long *>(ll_buf + slots_bytes) + 2;
    const unsigned long long epoch = *reinterpret_cast<volatile unsigned long long *>(mctr) + 1ull;
    const unsigned flag = (unsigned)epoch;
    const uint4 *slots = reinterpret_cast<const uint4 *>(ll_buf) + (size_t)(epoch & 1ull) * G * block_len;
    if (threadIdx.x == 0) { s_real = 0; s_hdr[0] = 0; s_hdr[1] = 0x7fffffffffffffffll; s_hdr[2] = 0; s_hdr[3] = 0; }
    __syncthreads();
    unsigned long long t0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    const int n = G * K;
    int my_real = 0;
    bool ok = true;
    // kLlBatch elements per thread are requested before any is examined (one L2 round trip per batch
    // when the data is already there); a slot that is not ready yet is polled again by ll_poll
    constexpr int kLlBatch = 4;
    for (int e0 = threadIdx.x; e0 < n; e0 += blockDim.x * kLlBatch) {
        uint4 wr[kLlBatch], wi[kLlBatch];
#pragma unroll
        for (int u = 0; u < kLlBatch; ++u) {
            const int e = e0 + u * blockDim.x;
            if (e < n) {
                const int g = e / K, i = e - g * K;
                const uint4 *blk = slots + (size_t)g * block_len;
                asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];"
                             : "=r"(wr[u].x), "=r"(wr[u].y), "=r"(wr[u].z), "=r"(wr[u].w) : "l"(blk + i) : "memory");
                asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];"
                             : "=r"(wi[u].x), "=r"(wi[u].y), "=r"(wi[u].z), "=r"(wi[u].w) : "l"(blk + K + i) : "memory");
            }
        }
#pragma unroll
        for (int u = 0; u < kLlBatch; ++u) {
            const int e = e0 + u * blockDim.x;
            if (e >= n) continue;
            const int g = e / K, i = e - g * K;
            const uint4 *blk = slots + (size_t)g * block_len;
            unsigned long long rc_bits = (unsigned long long)wr[u].x | ((unsigned long long)wr[u].z << 32);
            unsigned long long id_bits = (unsigned long long)wi[u].x | ((unsigned long long)wi[u].z << 32);
            if (wr[u].y != flag || wr[u].w != flag) ok = ll_poll(blk + i, flag, rc_bits, t0, timeout_ns) && ok;
            if (wi[u].y != flag || wi[u].w != flag) ok = ll_poll(blk + K + i, flag, id_bits, t0, timeout_ns) && ok;
            const long long id = (long long)id_bits;
            const KeyId v = (id < 0 || !ok) ? KeyId{~0ull, 0x7fffffffffffffffll}
                                            : KeyId{f64_to_sort_key(__longlong_as_double((long long)rc_bits)), id};
            stage[e] = v;
            my_real += v.key != ~0ull;
        }
    }
    if (blockIdx.x == 0) {
        my_real = warp_sum(my_real);
        if (lane_id() == 0 && my_real) atomicAdd(&s_real, my_real);
        for (int g = threadIdx.x; g < G; g += blockDim.x) {      // fold the per-rank pricing headers
            const uint4 *hdr = slots + (size_t)g * block_len + 2 * K;
            unsigned long long h0, h1, h3;
            ok = ll_poll(hdr, flag, h0, t0, timeout_ns) && ok;
            ok = ll_poll(hdr + 1, flag, h1, t0, timeout_ns) && ok;
            ok = ll_poll(hdr + 3, flag, h3, t0, timeout_ns) && ok;
            atomicAdd((unsigned long long *)&s_hdr[0], h0);
            atomicMin(&s_hdr[1], (long long)h1);
            atomicMax(&s_hdr[2], (long long)h0);
            atomicOr((unsigned long long *)&s_hdr[3], h3);
        }
    }
    if (!ok) atomicExch(status, SX_ERR_PEER_TIMEOUT);
    __syncthreads();
    if (blockIdx.x == 0) {
        const int n_out = s_real < K ? s_real : K;
        for (int i = n_out + threadIdx.x; i < K; i += blockDim.x) { out_rc[i] = INFINITY; out_id[i] = -1; }
        if (threadIdx.x == 0) {
            *out_n = n_out;
            if (out_summary) { out_summary[0] = s_hdr[0]; out_summary[1] = s_hdr[1]; out_summary[2] = s_hdr[2]; out_summary[3] = s_hdr[3]; }
        }
    }
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
        const int g = e / K, i = e - g * K;
        const KeyId mine = stage[e];
        if (mine.key == ~0ull) continue;
        int rank = i;
        for (int h = 0; h < G && rank < K; ++h) {
            if (h == g) continue;
            int lo = 0, hi = K;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (keyid_less(stage[h * K + mid], mine)) lo = mid + 1; else hi = mid;
            }
            rank += lo;
        }
        if (rank < K) { out_rc[rank] = sort_key_to_f64(mine.key); out_id[rank] = mine.id; }
    }
    // not done before the kernel this one was (programmatically) serialised after: what follows in the
    // stream may rely on both
    asm volatile("griddepcontrol.wait;" ::: "memory");
    __syncthreads();
    if (threadIdx.x == 0) {                       // the last CTA to finish advances the merge epoch
        __threadfence();
        if (atomicAdd(mctr + 1, 1ull) == (unsigned long long)(gridDim.x - 1)) {
            mctr[1] = 0ull;
            *reinterpret_cast<volatile unsigned long long *>(mctr) = epoch;
        }
    }
}

// ---- large-K path helpers ---------------------------------------------------------------
__global__ void tk_gather_kernel(const double *__restrict__ rc, const long long *__restrict__ id,
                                 const uint32_t *__restrict__ perm, long long n, double *rc_out, long long *id_out) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x) {
        const uint32_t s = perm[i];
        rc_out[i] = rc[s];
        id_out[i] = id[s];
    }
}
__global__ void tk_emit_kernel(const double *__restrict__ rc, const long long *__restrict__ id,
                               const uint32_t *__restrict__ perm, long long n, long long K, double *out_rc,
                               long long *out_id, long long *out_n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < K;
         i += (long long)gridDim.x * blockDim.x) {
        if (i < n) { const uint32_t s = perm[i]; out_rc[i] = rc[s]; out_id[i] = id[s]; }
        else { out_rc[i] = INFINITY; out_id[i] = -1; }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *out_n = n < K ? n : K;
}

static int tk_grid(long long n, int threads) {
    long long g = (n + threads - 1) / threads;
    if (g > num_sms() * 8) g = num_sms() * 8;
    if (g < 1) g = 1;
    return (int)g;
}

}  // namespace sx

using namespace sx;

extern "C" size_t sx_topk_workspace_bytes(int64_t cand_cap, int64_t K) {
    if (cand_cap < 0 || K < 0) return 0;
    const size_t fast = carve_bytes((size_t)kSurvCap, 16) + 2 * carve_bytes((size_t)(cand_cap > 0 ? cand_cap : 1), 16);
    if (K <= SX_TOPK_MAX_K) return fast + 256;
    return fast + 2 * carve_bytes((size_t)cand_cap, 8) + 2 * carve_bytes((size_t)cand_cap, 4) +
           sx_argsort_workspace_bytes(cand_cap) + 256;
}

// K > SX_TOPK_MAX_K: two stable radix argsorts over the candidates, by id, then by rc.  The candidate count
// is needed on the host to size the sorts (one stream synchronisation).  cv continues after the buffers of
// the K <= SX_TOPK_MAX_K selection.
static int topk_select_large_k(const double *cand_rc, const int64_t *cand_id, int64_t cand_cap, const SelState *sel,
                               int64_t K, double *out_rc, int64_t *out_id, int64_t *out_n, Carver &cv,
                               size_t ws_bytes, cudaStream_t st) {
    unsigned long long n64 = 0;
    SX_CUDA(cudaMemcpyAsync(&n64, &sel->n_cand, sizeof(n64), cudaMemcpyDeviceToHost, st));
    SX_CUDA(cudaStreamSynchronize(st));
    const long long n = n64 > (unsigned long long)cand_cap ? cand_cap : (long long)n64;
    double *rc1 = cv.take<double>(cand_cap);
    long long *id1 = cv.take<long long>(cand_cap);
    uint32_t *perm1 = cv.take<uint32_t>(cand_cap);
    uint32_t *perm2 = cv.take<uint32_t>(cand_cap);
    void *sort_ws = cv.base + cv.off;
    const size_t sort_ws_bytes = ws_bytes - cv.off;
    if (n > 0) {
        int rc = sx_argsort_u64((const unsigned long long *)cand_id, n, 63, perm1, nullptr, sort_ws, sort_ws_bytes, st);
        if (rc != SX_OK) return rc;
        tk_gather_kernel<<<tk_grid(n, 256), 256, 0, st>>>(cand_rc, (const long long *)cand_id, perm1, n, rc1, id1);
        SX_LAUNCH_CHECK();
        rc = sx_argsort_f64(rc1, n, perm2, nullptr, sort_ws, sort_ws_bytes, st);
        if (rc != SX_OK) return rc;
    }
    tk_emit_kernel<<<tk_grid(K, 256), 256, 0, st>>>(rc1, id1, perm2, n, K, out_rc, (long long *)out_id, (long long *)out_n);
    SX_LAUNCH_CHECK();
    return SX_OK;
}

extern "C" int sx_topk_select(const double *cand_rc, const int64_t *cand_id, int64_t cand_cap,
                              sx_select_state *sel, sx_price_header *header, int64_t K, double *out_rc,
                              int64_t *out_id, int64_t *out_n, void *ws, size_t ws_bytes, void *stream) {
    if (K <= 0 || cand_cap < 0 || !sel || !header || !out_rc || !out_id || !out_n) return SX_ERR_INVALID;
    if (cand_cap > 0 && (!cand_rc || !cand_id)) return SX_ERR_INVALID;
    if (!ws || ws_bytes < sx_topk_workspace_bytes(cand_cap, K)) return SX_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    SelState *sst = (SelState *)sel;
    Carver cv(ws);
    KeyId *sure = cv.take<KeyId>(kSurvCap);
    KeyId *listA = cv.take<KeyId>(cand_cap > 0 ? cand_cap : 1);
    KeyId *listB = cv.take<KeyId>(cand_cap > 0 ? cand_cap : 1);
    if (K > SX_TOPK_MAX_K)
        return topk_select_large_k(cand_rc, cand_id, cand_cap, sst, K, out_rc, out_id, out_n, cv, ws_bytes, st);
    const long long *cid = (const long long *)cand_id;
    int Ki = (int)K;
    long long *oid = (long long *)out_id, *on = (long long *)out_n;
    void *args[] = {(void *)&cand_rc, (void *)&cid, (void *)&cand_cap, (void *)&sst, (void *)&header, (void *)&Ki,
                    (void *)&sure, (void *)&listA, (void *)&listB, (void *)&out_rc, (void *)&oid, (void *)&on};
    SX_CUDA(cudaLaunchCooperativeKernel((void *)topk_select_kernel, dim3(num_sms()), dim3(kApThreads), args, 0, st));
    return SX_OK;
}

extern "C" size_t sx_topk_merge_workspace_bytes(int64_t G) {
    if (G < 0) return 0;
    return 2 * carve_bytes((size_t)G + 2, 4) + 256;
}

extern "C" int sx_topk_merge(const double *blocks_rc, const int64_t *blocks_id, int64_t block_stride, int64_t G,
                             int64_t K, const int64_t *headers, double *out_rc, int64_t *out_id, int64_t *out_n,
                             int64_t *out_summary, const unsigned long long *parity_ctr, int64_t parity_stride,
                             void *ws, size_t ws_bytes, void *stream) {
    if (G <= 0 || K <= 0 || !blocks_rc || !blocks_id || !out_rc || !out_id || !out_n) return SX_ERR_INVALID;
    if (parity_ctr && G * K > (1 << 22)) return SX_ERR_TOO_LARGE;
    if (block_stride < K || ((headers == nullptr) != (out_summary == nullptr))) return SX_ERR_INVALID;
    if (G > (1 << 20) || K > (1ll << 30)) return SX_ERR_TOO_LARGE;
    if (!ws || ws_bytes < sx_topk_merge_workspace_bytes(G)) return SX_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    if (G * K <= (1 << 22)) {
        const size_t stage_bytes = (size_t)G * K * sizeof(KeyId);
        const int use_smem = stage_bytes <= 200 * 1024;
        const int threads = use_smem ? 1024 : 256;
        long long mg = (G * K + threads - 1) / threads;
        if (mg > num_sms() * 4) mg = num_sms() * 4;
        if (use_smem) SX_CUDA(cudaFuncSetAttribute(merge_rank_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        merge_rank_kernel<<<(int)mg, threads, use_smem ? stage_bytes : 0, st>>>(blocks_rc, (const long long *)blocks_id, block_stride, (int)G,
                                                          (int)K, (const long long *)headers, out_rc,
                                                          (long long *)out_id, (long long *)out_n,
                                                          (long long *)out_summary, parity_ctr, parity_stride,
                                                          use_smem);
        SX_LAUNCH_CHECK();
        return SX_OK;
    }
    Carver cv(ws);
    int *plen = cv.take<int>(G + 2), *poff = cv.take<int>(G + 2);
    topk_prep_kernel<<<1, 1024, 0, st>>>(blocks_rc, (const long long *)blocks_id, block_stride, (int)G, (int)K, plen,
                                         poff, out_rc, (long long *)out_id, (long long *)out_n,
                                         (const long long *)headers, (long long *)out_summary);
    SX_LAUNCH_CHECK();
    topk_rank_kernel<<<num_sms() * 2, 256, 0, st>>>(blocks_rc, (const long long *)blocks_id, block_stride, (int)G, (int)K,
                                                  plen, poff, out_rc, (long long *)out_id);
    SX_LAUNCH_CHECK();
    return SX_OK;
}

extern "C" int sx_topk_merge_ll(void *ll_buf_local, int64_t block_len, int64_t G, int64_t K, double *out_rc,
                                int64_t *out_id, int64_t *out_n, int64_t *out_summary, int32_t *status_dev,
                                void *stream) {
    if (!ll_buf_local || G <= 0 || K <= 0 || block_len < 2 * K + 4 || !out_rc || !out_id || !out_n || !status_dev)
        return SX_ERR_INVALID;
    const size_t stage_bytes = (size_t)G * K * sizeof(KeyId);
    if (stage_bytes > 200 * 1024) return SX_ERR_TOO_LARGE;
    SX_CUDA(cudaFuncSetAttribute(merge_ll_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    long long mg = (G * K + 1023) / 1024;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)mg);
    cfg.blockDim = dim3(1024);
    cfg.dynamicSmemBytes = stage_bytes;
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    SX_CUDA(cudaLaunchKernelEx(&cfg, merge_ll_kernel, (char *)ll_buf_local, (long long)block_len, (int)G, (int)K, out_rc,
                               (long long *)out_id, (long long *)out_n, (long long *)out_summary, (int *)status_dev,
                               /*timeout_ns=*/10ull * 1000 * 1000 * 1000));
    return SX_OK;
}

// sx_merge.cuh -- merge of G sorted, padded per-rank top-K blocks into the global top-K (sm_100a).  The one
// definition behind sx_topk_merge (sx_topk.cu), sx_topk_merge_ll (sx_topk.cu) and the in-kernel merge of the
// fused pricing pass (sx_fused.cu).
//
// Every block holds K entries sorted by (rc, id), the real ones first and padding (+inf, -1) after them.  An
// element's position in the merged order is its index in its own block plus, for every other block, the
// number of entries below it: a binary search over the keys (f64_to_sort_key images), and only where the keys
// are equal a second one over the ids (ids are distinct across blocks).  Padding is an entry with id < 0, or
// with rc = +inf where only rc is read: real entries are violators, so never +inf, and padding sorts last.
#pragma once
#include "sx_ll.cuh"

namespace sx {

// Per-CTA fold (shared memory) of the G pricing headers and of the number of real entries.
struct MergeFold {
    long long hdr[4];      // total n_violating, min key, largest single n_violating, OR of the status words
    int       real;
};

__device__ __forceinline__ void merge_fold_init(MergeFold &s) {
    if (threadIdx.x == 0) { s.real = 0; s.hdr[0] = 0; s.hdr[1] = 0x7fffffffffffffffll; s.hdr[2] = 0; s.hdr[3] = 0; }
}
// called by every thread of a warp
__device__ __forceinline__ void merge_fold_real(MergeFold &s, int real) {
    real = warp_sum(real);
    if (lane_id() == 0 && real) atomicAdd(&s.real, real);
}
// header words {n_violating, min_rc_key, -, status} of one block
__device__ __forceinline__ void merge_fold_header(MergeFold &s, unsigned long long h0, unsigned long long h1,
                                                  unsigned long long h3) {
    atomicAdd((unsigned long long *)&s.hdr[0], h0);
    atomicMin(&s.hdr[1], (long long)h1);
    atomicMax(&s.hdr[2], (long long)h0);
    atomicOr((unsigned long long *)&s.hdr[3], h3);
}
// After a __syncthreads behind the folds: the outputs past n_out = min(real, K) become padding; out_n and, when
// given, the summary are written.  The rank step fills [0, n_out).
__device__ __forceinline__ void merge_write_tail(const MergeFold &s, int K, long long *out_rc_bits, long long *out_id,
                                                 long long *out_n, long long *out_summary) {
    const int n_out = s.real < K ? s.real : K;
    for (int i = n_out + threadIdx.x; i < K; i += blockDim.x) { out_rc_bits[i] = 0x7ff0000000000000ll; out_id[i] = -1; }
    if (threadIdx.x == 0) {
        *out_n = n_out;
        if (out_summary)
            for (int j = 0; j < 4; ++j) out_summary[j] = s.hdr[j];
    }
}

// Position in the merged order of the real element (key, id) at index i of block g; K or more when it is not
// among the K best.  key_at(h, j) / id_at(h, j) read entry j of block h; ids are read only where keys tie.
template <class KeyAt, class IdAt>
__device__ __forceinline__ int merge_rank(unsigned long long key, long long id, int g, int i, int G, int K,
                                          KeyAt key_at, IdAt id_at) {
    int rank = i;
    for (int h = 0; h < G && rank < K; ++h) {
        if (h == g) continue;
        int lo = 0, hi = K;                                            // first index with key >= mine
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (key_at(h, mid) < key) lo = mid + 1; else hi = mid; }
        if (lo < K && key_at(h, lo) == key) {
            // equal reduced costs in another block: the arc id decides
            int ub = lo, hi2 = K;                                      // first index with key > mine
            while (ub < hi2) { const int mid = (ub + hi2) >> 1; if (key_at(h, mid) <= key) ub = mid + 1; else hi2 = mid; }
            int a = lo, b = ub;                                        // first index in [lo, ub) with id >= mine
            while (a < b) { const int mid = (a + b) >> 1; if (id_at(h, mid) < id) a = mid + 1; else b = mid; }
            lo = a;
        }
        rank += lo;
    }
    return rank;
}

// Merge of the G blocks of `epoch` out of the local LL exchange buffer `buf` (sx_ll.cuh) by n_merge CTAs, of
// which this one is number mc.  Every merge CTA stages the keys of all G blocks in mkey (G * K words of shared
// memory) as they land -- staging is the wait -- and ranks a contiguous range of the elements; CTA 0 also folds
// the headers and writes the padding, out_n and the summary.  false: a slot did not arrive within timeout_ns.
__device__ __forceinline__ bool merge_ll(char *buf, long long block_len, int G, int K, unsigned long long epoch,
                                         int mc, int n_merge, unsigned long long *mkey, MergeFold &s,
                                         long long *out_rc_bits, long long *out_id, long long *out_n,
                                         long long *out_summary, unsigned long long timeout_ns) {
    const int tid = threadIdx.x, nthr = blockDim.x;
    const unsigned flag = (unsigned)epoch;
    const int GK = G * K;
    const unsigned long long kPadKey = f64_to_sort_key(INFINITY);
    const unsigned long long t_start = global_timer_ns();
    bool ok = true;
    merge_fold_init(s);
    __syncthreads();                                                   // the caller's shared memory is free
    // elements of this CTA: [e_lo, e_hi), thread t takes e_lo + t, e_lo + t + nthr, ...  The id of the first one
    // is requested before the keys so that it is in flight with them.
    const int per_cta = (GK + n_merge - 1) / n_merge;
    const int e_lo = mc * per_cta, e_hi = (e_lo + per_cta < GK) ? e_lo + per_cta : GK;
    uint4 w_id = make_uint4(0u, 0u, 0u, 0u);
    if (e_lo + tid < e_hi) {
        const int g = (e_lo + tid) / K;
        w_id = ll_load_slot(ll_slot(buf, G, block_len, epoch, g, (long long)K + (e_lo + tid - g * K)));
    }
    {
        // kBatch slots are requested together and the whole batch is requested again until every slot carries
        // this epoch's flag: the merge CTAs start polling while the peers are still ranking, and re-polling the
        // late slots one by one would cost one L2 round trip each (28 per thread at G = 8: 20 us; measured).
        constexpr int kBatch = 8;
        int real = 0;
        for (int e0 = tid; e0 < GK; e0 += nthr * kBatch) {
            uint4 w[kBatch];
            for (;;) {
                bool all = true;
#pragma unroll
                for (int u = 0; u < kBatch; ++u) {
                    const int e = e0 + u * nthr;
                    if (e < GK) { const int g = e / K; w[u] = ll_load_slot(ll_slot(buf, G, block_len, epoch, g, e - g * K)); }
                }
#pragma unroll
                for (int u = 0; u < kBatch; ++u) {
                    const int e = e0 + u * nthr;
                    if (e < GK && !ll_ready(w[u], flag)) all = false;
                }
                if (all) break;
                if (global_timer_ns() - t_start > timeout_ns) { ok = false; break; }
            }
#pragma unroll
            for (int u = 0; u < kBatch; ++u) {
                const int e = e0 + u * nthr;
                if (e >= GK) continue;
                const unsigned long long bits = ll_ready(w[u], flag) ? ll_value(w[u]) : 0x7ff0000000000000ull;
                const unsigned long long key = f64_to_sort_key(__longlong_as_double((long long)bits));
                mkey[e] = key;
                real += key != kPadKey;
            }
        }
        if (mc == 0) {
            merge_fold_real(s, real);
            for (int g = tid; g < G; g += nthr) {
                unsigned long long h0, h1, h3;
                const uint4 *hdr = ll_slot(buf, G, block_len, epoch, g, (long long)2 * K);
                ok = ll_poll(hdr, flag, h0, t_start, timeout_ns) && ok;
                ok = ll_poll(hdr + 1, flag, h1, t_start, timeout_ns) && ok;
                ok = ll_poll(hdr + 3, flag, h3, t_start, timeout_ns) && ok;
                merge_fold_header(s, h0, h1, h3);
            }
        }
    }
    __syncthreads();
    if (mc == 0) merge_write_tail(s, K, out_rc_bits, out_id, out_n, out_summary);
    for (int my_e = e_lo + tid; my_e < e_hi; my_e += nthr) {
        const unsigned long long key = mkey[my_e];
        if (key == kPadKey) continue;
        const int my_g = my_e / K, my_i = my_e - my_g * K;
        unsigned long long id_bits = ll_value(w_id);
        if (my_e != e_lo + tid || !ll_ready(w_id, flag))
            ok = ll_poll(ll_slot(buf, G, block_len, epoch, my_g, (long long)K + my_i), flag, id_bits, t_start, timeout_ns) && ok;
        const long long my_id = (long long)id_bits;
        const int rank = merge_rank(
            key, my_id, my_g, my_i, G, K, [&](int h, int j) { return mkey[h * K + j]; },
            [&](int h, int j) {
                unsigned long long ob;
                ok = ll_poll(ll_slot(buf, G, block_len, epoch, h, (long long)K + j), flag, ob, t_start, timeout_ns) && ok;
                return (long long)ob;
            });
        if (rank < K) {
            out_rc_bits[rank] = __double_as_longlong(sort_key_to_f64(key));
            out_id[rank] = my_id;
        }
    }
    return ok;
}

}  // namespace sx

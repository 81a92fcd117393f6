// sx_topk.cu -- selection of the K most violating arcs (sm_100a).
//
// north_star extension (SURVEY.md section 8 row a9; the reference never ranks violators, it
// only tests `np.all(rc >= -tol)`, net_manager.py:318,496): among the candidates (rc, arc id)
// compacted by the pricing kernels, return the K smallest by (rc ascending, id ascending).
// (rc, id) is a strict total order, so the result does not depend on the (unordered)
// compaction or on how many GPUs priced the matrix.
//
// K <= 1024: ONE cooperative launch (topk_select_kernel), no host round trip.  It runs select_topk
// (sx_select.cuh), the same selection the fused pricing pass runs in its own kernel (sx_fused.cu):
//   1. filter: the pricing kernels left a histogram of the candidates' reduced costs; b* = the
//      smallest bin whose cumulative count reaches K.  Candidates with bin < b* are among the K
//      best, bin b* (0.4 % wide) is the boundary list;
//   2. refine: while the list is too long, an 11-bit digit of (key, id) splits the boundary list
//      again; a list of distinct (key, id) pairs shrinks to one element within 12 levels;
//   3. all-pairs rank: every survivor counts the survivors below it; that count is its
//      position in the output.  O(n_surv^2) compares spread over the whole GPU (1 to 32 lanes
//      per element), a few microseconds for the typical 1-2 K survivors.
//   The candidates must be distinct arcs.  Only copies of one (rc, id) pair -- the same arc priced
//   into one pass many times -- can keep the list long; the selection is then void and raises
//   SX_STATUS_DUPLICATE_CANDIDATES in the pricing header.
// K > 1024: two stable radix argsorts (by id, then by rc) over the candidates.
// Merge of G sorted, padded per-GPU lists after the exchange (sx_topk_merge, sx_topk_merge_ll): an element's
// position is the number of entries below it in every list, by the rank step, header fold and final write of
// sx_merge.cuh, which the in-kernel merge of the fused pass (sx_fused.cu) runs as well.  Above 2^22 elements a
// prefix bound over the (key, id) order first limits the elements that are ranked.
#include <math.h>

#include <cooperative_groups.h>

#include "sx_common.cuh"
#include "sx_select.cuh"
#include "sx_merge.cuh"

namespace cg = cooperative_groups;

namespace sx {

// (key, id) of entry `off` of a block; padding (id < 0) sorts last
__device__ __forceinline__ KeyId merge_load(const double *rc, const long long *id, long long off) {
    const long long i = id[off];
    return i < 0 ? KeyId{~0ull, 0x7fffffffffffffffll} : KeyId{f64_to_sort_key(rc[off]), i};
}
// entries of the sorted block prefix [0, len) below x (or_equal: not above x)
__device__ __forceinline__ int bound_list(const double *rc, const long long *id, int len, const KeyId &x, bool or_equal) {
    int lo = 0, hi = len;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const KeyId m = merge_load(rc, id, mid);
        if (or_equal ? !keyid_less(x, m) : keyid_less(m, x)) lo = mid + 1; else hi = mid;
    }
    return lo;
}
// real entries of the block prefix [0, len): the index of the first padding entry (ids are -1 from there on)
__device__ __forceinline__ int real_len(const long long *id, int len) {
    int lo = 0, hi = len;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (id[mid] >= 0) lo = mid + 1; else hi = mid; }
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
    __shared__ MergeFold s_fold;
    __shared__ KeyId s_thr[32];
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
    auto block_min_keyid = [&](KeyId c, bool want_max) -> KeyId {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const KeyId other{__shfl_xor_sync(0xffffffffu, c.key, o), __shfl_xor_sync(0xffffffffu, c.id, o)};
            if (keyid_less(other, c) != want_max) c = other;
        }
        __syncthreads();
        if (lane == 0) s_thr[warp] = c;
        __syncthreads();
        KeyId r = s_thr[0];
        for (int w = 1; w < 32; ++w) if (keyid_less(s_thr[w], r) != want_max) r = s_thr[w];
        return r;
    };
    merge_fold_init(s_fold);
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    // bound 1: the smallest "last element of a list" (padding: no constraint)
    KeyId thr{~0ull, 0x7fffffffffffffffll};
    long long n_real_lists = 0;
    for (int l = threadIdx.x; l < L; l += blockDim.x) {
        const KeyId c = merge_load(lists_rc, lists_id, (long long)l * LS + K - 1);
        if (keyid_less(c, thr)) thr = c;
        plen[l] = real_len(lists_id + (long long)l * LS, K);
        n_real_lists += plen[l];
    }
    thr = block_min_keyid(thr, false);
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
        KeyId deep{0ull, -1};                          // below every entry
        for (int l = threadIdx.x; l < L; l += blockDim.x) {
            const int take = plen[l] < lo ? plen[l] : lo;
            if (take > 0) {
                const KeyId c = merge_load(lists_rc, lists_id, (long long)l * LS + take - 1);
                if (keyid_less(deep, c)) deep = c;
            }
        }
        deep = block_min_keyid(deep, true);
        if (keyid_less(deep, thr)) thr = deep;
    }
    __syncthreads();
    // prefix lengths and their exclusive scan, 1024 lists per sweep
    long long real_total = 0;
    for (int base = 0; base < L; base += blockDim.x) {
        const int l = base + threadIdx.x;
        int len = 0;
        // without padding that ties with an all-padding threshold
        if (l < L) len = real_len(lists_id + (long long)l * LS, bound_list(lists_rc + (long long)l * LS, lists_id + (long long)l * LS, K, thr, true));
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
    if (headers)
        for (int l = threadIdx.x; l < L; l += blockDim.x) {
            const long long *h = headers + (long long)l * LS;
            merge_fold_header(s_fold, h[0], h[1], h[3]);
        }
    if (threadIdx.x == 0) { poff[L] = (int)real_total; s_fold.real = (int)real_total; }
    __syncthreads();
    // the rank kernel (next launch) writes the first out_n entries
    merge_write_tail(s_fold, K, reinterpret_cast<long long *>(out_rc), out_id, out_n, out_summary);
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
        const KeyId c = merge_load(lists_rc, lists_id, (long long)l * LS + i);
        int rank = 0;
        for (int m = lane; m < L; m += 32) {
            if (m == l) rank += i;
            else {
                const int len = plen[m];
                if (len) rank += bound_list(lists_rc + (long long)m * LS, lists_id + (long long)m * LS, len, c, false);
            }
        }
        rank = warp_sum(rank);
        if (lane == 0 && rank < K) { out_rc[rank] = lists_rc[(long long)l * LS + i]; out_id[rank] = c.id; }
    }
}

// ---- K <= SX_TOPK_MAX_K: select_topk (sx_select.cuh) in ONE cooperative launch ----
__global__ void __launch_bounds__(kSelThreads)
topk_select_kernel(const double *__restrict__ cand_rc, const long long *__restrict__ cand_id, long long cand_cap,
                   SelState *st, sx_price_header *hdr, int K, SelLists lists, double *__restrict__ out_rc,
                   long long *__restrict__ out_id, long long *out_n) {
    __shared__ SelScratch s;
    const unsigned long long n64 = st->n_cand;
    long long n = (long long)n64;
    if (n64 > (unsigned long long)cand_cap) {
        n = cand_cap;
        if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(&hdr->status, kStatusCandOverflow);
    }
    // the candidate list was pruned for the K given to sx_price_pass_begin: a larger K here cannot be served
    if ((unsigned)K > st->K && blockIdx.x == 0 && threadIdx.x == 0) atomicOr(&hdr->status, kStatusKMismatch);
    const SelResult r = select_topk(
        cand_rc, cand_id, n, cand_cap, st, K, lists, s, [] { cg::this_grid().sync(); },
        [&](const KeyId &v, int rank, int sub, int) {
            if (sub == 0 && rank < K) {
                out_rc[rank] = sort_key_to_f64(v.key);
                out_id[rank] = v.id;
            }
        });
    if (blockIdx.x == 0) {
        for (int i = r.n_out + threadIdx.x; i < K; i += kSelThreads) { out_rc[i] = INFINITY; out_id[i] = -1; }
        if (threadIdx.x == 0) {
            *out_n = r.n_out;
            if (r.duplicates) atomicOr(&hdr->status, kStatusDuplicateCandidates);
        }
    }
}

// Merge of G sorted, padded blocks of K (exchanged between G ranks): one thread per element, ranked by
// merge_rank (sx_merge.cuh).  The keys of every block are staged in shared memory when they fit (coalesced
// loads, then ~G * 10 shared loads per element); otherwise the blocks are searched in global memory.
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
    extern __shared__ __align__(16) unsigned char mg_raw[];
    unsigned long long *mkey = reinterpret_cast<unsigned long long *>(mg_raw);
    __shared__ MergeFold s_fold;
    merge_fold_init(s_fold);
    if (use_smem)
        for (int e = threadIdx.x; e < n; e += blockDim.x) {
            const int g = e / K;
            mkey[e] = f64_to_sort_key(blocks_rc[(long long)g * LS + (e - g * K)]);
        }
    __syncthreads();
    if (blockIdx.x == 0) {
        int real = 0;
        for (int g = threadIdx.x; g < G; g += blockDim.x) {
            real += real_len(blocks_id + (long long)g * LS, K);
            if (headers) { const long long *h = headers + (long long)g * LS; merge_fold_header(s_fold, h[0], h[1], h[3]); }
        }
        merge_fold_real(s_fold, real);
        __syncthreads();
        merge_write_tail(s_fold, K, reinterpret_cast<long long *>(out_rc), out_id, out_n, out_summary);
    }
    const auto key_at = [&](int h, int j) {
        return use_smem ? mkey[h * K + j] : f64_to_sort_key(blocks_rc[(long long)h * LS + j]);
    };
    const auto id_at = [&](int h, int j) { return blocks_id[(long long)h * LS + j]; };
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
        const int g = e / K, i = e - g * K;
        const long long id = id_at(g, i);
        if (id < 0) continue;                                  // padding
        const int rank = merge_rank(key_at(g, i), id, g, i, G, K, key_at, id_at);
        if (rank < K) { out_rc[rank] = blocks_rc[(long long)g * LS + i]; out_id[rank] = id; }
    }
}

// Merge straight out of the LL exchange buffer (sx_exchange_push_ll) by merge_ll (sx_merge.cuh), with all CTAs
// of the grid: staging a block in shared memory IS the wait for it.
__global__ void __launch_bounds__(1024)
merge_ll_kernel(char *ll_buf, long long block_len, int G, int K, double *__restrict__ out_rc,
                long long *__restrict__ out_id, long long *out_n, long long *out_summary, int *status,
                unsigned long long timeout_ns) {
    extern __shared__ __align__(16) unsigned char mg_raw[];
    __shared__ MergeFold s_fold;
    // The merge keeps an epoch counter of its own ([2], [3] = CTAs done), advanced once per launch like the
    // pushing side's ([0], [1]): it depends on no other kernel of this GPU, so it may be launched with
    // programmatic stream serialisation and become resident while the pricing kernel is still draining.
    unsigned long long *mctr = ll_counters(ll_buf, G, block_len) + 2;
    const unsigned long long epoch = *reinterpret_cast<volatile unsigned long long *>(mctr) + 1ull;
    if (!merge_ll(ll_buf, block_len, G, K, epoch, blockIdx.x, gridDim.x, reinterpret_cast<unsigned long long *>(mg_raw),
                  s_fold, reinterpret_cast<long long *>(out_rc), out_id, out_n, out_summary, timeout_ns))
        atomicExch(status, SX_ERR_PEER_TIMEOUT);
    // not done before the kernel this one was (programmatically) serialised after: what follows in the
    // stream may rely on both
    asm volatile("griddepcontrol.wait;" ::: "memory");
    __syncthreads();
    if (threadIdx.x == 0) advance_epoch_when_last(mctr, gridDim.x, epoch);
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
    SelLists lists = carve_sel_lists(cv, cand_cap);
    if (K > SX_TOPK_MAX_K)
        return topk_select_large_k(cand_rc, cand_id, cand_cap, sst, K, out_rc, out_id, out_n, cv, ws_bytes, st);
    const long long *cid = (const long long *)cand_id;
    int Ki = (int)K;
    long long *oid = (long long *)out_id, *on = (long long *)out_n;
    void *args[] = {(void *)&cand_rc, (void *)&cid, (void *)&cand_cap, (void *)&sst, (void *)&header, (void *)&Ki,
                    (void *)&lists, (void *)&out_rc, (void *)&oid, (void *)&on};
    SX_CUDA(cudaLaunchCooperativeKernel((void *)topk_select_kernel, dim3(num_sms()), dim3(kSelThreads), args, 0, st));
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
        const size_t stage_bytes = (size_t)G * K * sizeof(unsigned long long);
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
    if ((size_t)G * K * 16 > 200 * 1024) return SX_ERR_TOO_LARGE;     // the ABI limit (keys and ids once)
    const size_t stage_bytes = (size_t)G * K * sizeof(unsigned long long);
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

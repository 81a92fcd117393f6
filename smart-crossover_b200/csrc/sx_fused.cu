// sx_fused.cu -- one launch per pricing pass: price + select + exchange + merge (sm_100a).
//
// A column-generation pricing pass (reference net_manager.py:474-497, plus the north_star top-k) used to
// be five launches on the critical path -- pass begin (state clear), pricing, cooperative selection, push
// of the result block to the peer GPUs, merge -- and on a row slab of a few hundred MB their launch gaps
// and grid-wide barriers cost as much as the pricing itself.  price_fused_kernel does all of it:
//
//   start    every CTA clears its slice of the OTHER selection state (the pricer owns two, used by
//            alternate passes), so no pass ever waits for a clear;
//   pricing  the TMA pipeline of sx_price_tma.cuh, unchanged: count, min, candidate list + histogram;
//   barrier  grid-wide (the kernel is launched cooperatively: all CTAs are resident);
//   select   select_topk (sx_select.cuh), the selection topk_select_kernel runs too: a candidate list of at
//            most kDirectCap is ranked as it is; a longer one is first split by the histogram's bound b*
//            (every CTA derives it: one warp, 9 KB of L2 reads) into the sure candidates and the boundary
//            list, which radix refinement shortens further only under massive ties at the K-th value;
//            second barrier;
//   rank     all-pairs rank of the candidates / survivors spread over the grid (1-32 lanes per element);
//            the lanes of an element write it to its position in the local result block AND, with G > 1,
//            store it as flag-in-data slots straight into every peer's exchange buffer (NVLink; sx_ll.cuh),
//            so the exchange needs no kernel of its own and starts while other elements are still ranked;
//   merge    (G > 1) the last CTAs of the grid -- which have no rank work -- stage the keys of all G blocks
//            out of the local exchange buffer as they land (staging is the wait), rank every element by
//            G - 1 binary searches in shared memory and write the merged top-K.
//
// If the candidate buffer overflowed, the pass raises SX_STATUS_CAND_OVERFLOW in the header -- it still
// pushes a well-formed block so that no peer waits -- and the caller grows the buffer and repeats the pass.
#include <stdlib.h>

#include "sx_gridbar.cuh"
#include "sx_ll.cuh"
#include "sx_price_tma.cuh"

namespace sx {

constexpr int kMergeCtas = 64;          // CTAs (from the end of the grid) that merge the G blocks

struct FusedCtl {
    unsigned long long pass;      // passes completed; parity selects the selection state in use
    GridBarrier        bar;       // grid-wide barrier (sx_gridbar.cuh)
    unsigned int       dyn_ctr;   // tail stealing of the pricing walk: next dynamically assigned tile (0 between passes)
    unsigned int       pad[3];
    unsigned long long ts[8];     // diagnostics: %globaltimer of CTA 0 at the phase boundaries of the last pass
};
struct FusedState {
    SelState sel[2];
    FusedCtl ctl;
};
static_assert(sizeof(FusedState) % 16 == 0, "");

struct FusedParams {
    FusedState      *state;
    const double    *cand_rc;
    const long long *cand_id;
    long long        cand_cap;
    unsigned         K;              // >= 1 (layout); cand_cap == 0 means count / min only
    long long       *block;          // local result block [K rc bits | K ids | header (4) | n_out | pad]
    SelLists         lists;          // lists of the selection (workspace of sx_topk_workspace_bytes)
    char *const     *peer_bufs;      // LL exchange buffers of the G ranks, or nullptr (no exchange)
    int              rank, G;
    long long        block_len;
    // in-kernel merge (peer_bufs != nullptr and merged != nullptr)
    long long       *merged;         // [K rc bits | K ids | n_out | total count, min key, largest count, status]
    int             *xstatus;        // SX_ERR_PEER_TIMEOUT lands here
    unsigned long long timeout_ns;
    int              steal;          // 1: the last eighth of the tiles is handed out dynamically
};

__device__ __forceinline__ unsigned long long ld_volatile_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void stamp(FusedCtl *ctl, int i) {
    if (blockIdx.x == 0 && threadIdx.x == 0) ctl->ts[i] = global_timer_ns();
}

// slot `idx` of rank r's block, parity half of `epoch`, in the exchange buffer `buf`
__device__ __forceinline__ uint4 *ll_slot(char *buf, const FusedParams &f, unsigned long long epoch, int r, long long idx) {
    return reinterpret_cast<uint4 *>(buf) + ((size_t)(epoch & 1ull) * f.G + r) * f.block_len + idx;
}

template <int ROWS, int STAGES, int CWARPS, int MINB>
__global__ void __launch_bounds__((CWARPS + 1) * 32, MINB)
price_fused_kernel(const __grid_constant__ CUtensorMap tmap, const DenseParams p0, const FusedParams f) {
    static_assert((size_t)STAGES * ROWS * kBoxCols * sizeof(double) >= sizeof(SelScratch),
                  "the stage ring is reused as the selection's shared memory");
    static_assert(CWARPS * 32 == kSelThreads, "the consumer warps select, the producer warp joins the barriers");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ long long s_hdr[4];
    __shared__ int s_real;
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int K = (int)f.K;
    FusedCtl *ctl = &f.state->ctl;
    const unsigned long long pass = ld_volatile_u64(&ctl->pass);
    SelState *sel = &f.state->sel[pass & 1ull];
    SelState *nxt = &f.state->sel[(pass & 1ull) ^ 1ull];
    if (blockIdx.x == 0 && tid == 0) ctl->ts[7] = ctl->ts[6];     // end of the previous pass (its last CTA)
    stamp(ctl, 0);
    unsigned long long epoch = 0, *ll_ctr = nullptr;
    char *ll_local = nullptr;
    if (f.peer_bufs) {
        ll_local = f.peer_bufs[f.rank];
        ll_ctr = reinterpret_cast<unsigned long long *>(ll_local + (size_t)2 * f.G * f.block_len * 16);
        epoch = ld_volatile_u64(ll_ctr) + 1ull;
    }
    const unsigned flag = (unsigned)epoch;
    // ---- clear the other selection state for the next pass ----
    {
        uint4 *w = reinterpret_cast<uint4 *>(nxt);
        const size_t n16 = sizeof(SelState) / 16;
        for (size_t i = (size_t)blockIdx.x * nthr + tid; i < n16; i += (size_t)gridDim.x * nthr)
            w[i] = sel_clear_word(i, f.K);
    }
    // ---- pricing ----
    DenseParams p = p0;
    p.sink.hdr = &sel->hdr;
    p.sink.sel = sel;
    p.dyn_ctr = f.steal ? &ctl->dyn_ctr : nullptr;
    price_tiles<ROWS, STAGES, CWARPS, false>(tmap, p, smem_raw);
    stamp(ctl, 1);

    grid_barrier(&ctl->bar);      // header, histogram and candidate list of this pass are complete
    stamp(ctl, 2);
    if (blockIdx.x == 0 && tid == 0) {
        // every CTA has read `pass` and the exchange epoch: advance them for the next launch (the merge
        // epoch [2] moves with the push epoch [0]: this kernel is both sides of the exchange)
        *reinterpret_cast<volatile unsigned long long *>(&ctl->pass) = pass + 1ull;
        *reinterpret_cast<volatile unsigned int *>(&ctl->dyn_ctr) = 0u;      // every CTA is past its pricing walk
        if (ll_ctr) {
            *reinterpret_cast<volatile unsigned long long *>(ll_ctr) = epoch;
            if (f.merged) *reinterpret_cast<volatile unsigned long long *>(ll_ctr + 2) = epoch;
        }
    }

    const unsigned long long n64 = __ldcg(&sel->n_cand);
    const long long n = n64 > (unsigned long long)f.cand_cap ? f.cand_cap : (long long)n64;
    // ---- selection; the lanes of an element emit it ----
    stamp(ctl, 3);        // a list ranked as it is has no second barrier; a longer one stamps 3 and 4 around it
    stamp(ctl, 4);
    const SelResult sr = select_topk(
        f.cand_rc, f.cand_id, n, f.cand_cap, sel, K, f.lists, *reinterpret_cast<SelScratch *>(smem_raw),
        [ctl] { stamp(ctl, 3); grid_barrier(&ctl->bar); stamp(ctl, 4); },
        [&](const KeyId &v, int rank, int sub, int L) {
            if (rank >= K) return;
            const unsigned long long rc_bits = (unsigned long long)__double_as_longlong(sort_key_to_f64(v.key));
            if (sub == 0) { f.block[rank] = (long long)rc_bits; f.block[K + rank] = v.id; }
            if (f.peer_bufs)
                for (int q = sub; q < f.G; q += L) {
                    ll_store_slot(ll_slot(f.peer_bufs[q], f, epoch, f.rank, rank), flag, rc_bits);
                    ll_store_slot(ll_slot(f.peer_bufs[q], f, epoch, f.rank, (long long)K + rank), flag,
                                  (unsigned long long)v.id);
                }
        });
    const int n_out = sr.n_out;
    stamp(ctl, 5);

    // ---- padding, header and count: the last CTA (it rarely has rank work) ----
    if (blockIdx.x == gridDim.x - 1) {
        const unsigned long long pad_rc = 0x7ff0000000000000ull;    // +inf
        for (int i = n_out + tid; i < K; i += nthr) {
            f.block[i] = (long long)pad_rc; f.block[K + i] = -1;
            if (f.peer_bufs)
                for (int q = 0; q < f.G; ++q) {
                    ll_store_slot(ll_slot(f.peer_bufs[q], f, epoch, f.rank, i), flag, pad_rc);
                    ll_store_slot(ll_slot(f.peer_bufs[q], f, epoch, f.rank, (long long)K + i), flag, ~0ull);
                }
        }
        if (tid < 6) {
            unsigned long long w = 0;
            if (tid == 0) w = __ldcg(&sel->hdr.n_violating);
            if (tid == 1) w = (unsigned long long)__ldcg(&sel->hdr.min_rc_key);
            if (tid == 2) w = __ldcg(&sel->hdr.n_priced);
            if (tid == 3)
                w = __ldcg(&sel->hdr.status) | (n64 > (unsigned long long)f.cand_cap ? kStatusCandOverflow : 0ull) |
                    (sr.duplicates ? kStatusDuplicateCandidates : 0ull);
            if (tid == 4) w = (unsigned long long)n_out;
            f.block[2 * K + tid] = (long long)w;
            if (f.peer_bufs)
                for (int q = 0; q < f.G; ++q)
                    ll_store_slot(ll_slot(f.peer_bufs[q], f, epoch, f.rank, (long long)2 * K + tid), flag, w);
        }
    }

    if (blockIdx.x == gridDim.x - 1 && tid == 0) ctl->ts[6] = global_timer_ns();   // overwritten at the end of the merge
    // ---- merge of the G blocks out of the local exchange buffer (replaces sx_topk_merge_ll) ----
    if (f.peer_bufs == nullptr || f.merged == nullptr) return;
    const int n_merge = gridDim.x < kMergeCtas ? (int)gridDim.x : kMergeCtas;
    const int mc = (int)blockIdx.x - ((int)gridDim.x - n_merge);           // index among the merge CTAs
    if (mc < 0) return;
    const int GK = f.G * K;
    unsigned long long *mkey = reinterpret_cast<unsigned long long *>(smem_raw);   // GK keys; padding = key(+inf)
    const unsigned long long kPadKey = f64_to_sort_key(INFINITY);
    const unsigned long long t_start = global_timer_ns();
    bool ok = true;
    if (tid == 0) { s_real = 0; s_hdr[0] = 0; s_hdr[1] = 0x7fffffffffffffffll; s_hdr[2] = 0; s_hdr[3] = 0; }
    __syncthreads();                                                       // the rank tiles are no longer read
    // elements of this CTA: [e_lo, e_hi), thread t takes e_lo + t, e_lo + t + nthr, ...  The id of the first one
    // is requested before the keys so that it is in flight with them.
    const int per_cta = (GK + n_merge - 1) / n_merge;
    const int e_lo = mc * per_cta, e_hi = (e_lo + per_cta < GK) ? e_lo + per_cta : GK;
    uint4 w_id = make_uint4(0u, 0u, 0u, 0u);
    if (e_lo + tid < e_hi) {
        const int g = (e_lo + tid) / K;
        w_id = ll_load_slot(ll_slot(ll_local, f, epoch, g, (long long)K + (e_lo + tid - g * K)));
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
                    if (e < GK) { const int g = e / K; w[u] = ll_load_slot(ll_slot(ll_local, f, epoch, g, e - g * K)); }
                }
#pragma unroll
                for (int u = 0; u < kBatch; ++u) {
                    const int e = e0 + u * nthr;
                    if (e < GK && !ll_ready(w[u], flag)) all = false;
                }
                if (all) break;
                if (global_timer_ns() - t_start > f.timeout_ns) { ok = false; break; }
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
        if (mc == 0) {                                                     // one CTA folds the headers and the count
            real = warp_sum(real);
            if (lane_id() == 0 && real) atomicAdd(&s_real, real);
            for (int g = tid; g < f.G; g += nthr) {
                unsigned long long h0, h1, h3;
                ok = ll_poll(ll_slot(ll_local, f, epoch, g, (long long)2 * K), flag, h0, t_start, f.timeout_ns) && ok;
                ok = ll_poll(ll_slot(ll_local, f, epoch, g, (long long)2 * K + 1), flag, h1, t_start, f.timeout_ns) && ok;
                ok = ll_poll(ll_slot(ll_local, f, epoch, g, (long long)2 * K + 3), flag, h3, t_start, f.timeout_ns) && ok;
                atomicAdd((unsigned long long *)&s_hdr[0], h0);
                atomicMin(&s_hdr[1], (long long)h1);
                atomicMax(&s_hdr[2], (long long)h0);
                atomicOr((unsigned long long *)&s_hdr[3], h3);
            }
        }
    }
    __syncthreads();
    if (mc == 0) {
        const int n_tot = s_real < K ? s_real : K;
        for (int i = n_tot + tid; i < K; i += nthr) { f.merged[i] = 0x7ff0000000000000ll; f.merged[K + i] = -1; }
        if (tid == 0) {
            f.merged[2 * K] = n_tot;
            f.merged[2 * K + 1] = s_hdr[0]; f.merged[2 * K + 2] = s_hdr[1];
            f.merged[2 * K + 3] = s_hdr[2]; f.merged[2 * K + 4] = s_hdr[3];
        }
    }
    for (int my_e = e_lo + tid; my_e < e_hi; my_e += nthr) {
        const unsigned long long key = mkey[my_e];
        if (key == kPadKey) continue;
        const int my_g = my_e / K, my_i = my_e - my_g * K;
        unsigned long long id_bits = ll_value(w_id);
        if (my_e != e_lo + tid || !ll_ready(w_id, flag))
            ok = ll_poll(ll_slot(ll_local, f, epoch, my_g, (long long)K + my_i), flag, id_bits, t_start, f.timeout_ns) && ok;
        const long long my_id = (long long)id_bits;
        int rank = my_i;
        for (int h = 0; h < f.G && rank < K; ++h) {
            if (h == my_g) continue;
            const unsigned long long *kh = mkey + h * K;
            int lo = 0, hi = K;                                            // first index with key >= mine
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (kh[mid] < key) lo = mid + 1; else hi = mid; }
            if (lo < K && kh[lo] == key) {
                // equal reduced costs in another block: the arc id decides; ids are read from the buffer
                int ub = lo, hi2 = K;                                      // first index with key > mine
                while (ub < hi2) { const int mid = (ub + hi2) >> 1; if (kh[mid] <= key) ub = mid + 1; else hi2 = mid; }
                int a = lo, b = ub;                                        // first index in [lo, ub) with id >= mine
                while (a < b) {
                    const int mid = (a + b) >> 1;
                    unsigned long long ob;
                    ok = ll_poll(ll_slot(ll_local, f, epoch, h, (long long)K + mid), flag, ob, t_start, f.timeout_ns) && ok;
                    if ((long long)ob < my_id) a = mid + 1; else b = mid;
                }
                lo = a;
            }
            rank += lo;
        }
        if (rank < K) {
            f.merged[rank] = __double_as_longlong(sort_key_to_f64(key));
            f.merged[K + rank] = my_id;
        }
    }
    if (!ok) atomicExch(f.xstatus, SX_ERR_PEER_TIMEOUT);
    if (mc == n_merge - 1 && tid == 0) ctl->ts[6] = global_timer_ns();      // end of the merge (diagnostics)
}

__global__ void __launch_bounds__(256) fused_init_kernel(FusedState *st, unsigned K) {
    const size_t n16 = sizeof(SelState) / 16;
    for (int h = 0; h < 2; ++h) {
        uint4 *w = reinterpret_cast<uint4 *>(&st->sel[h]);
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x)
            w[i] = sel_clear_word(i, K);
    }
    static_assert(sizeof(FusedCtl) / 4 <= 256, "");
    if (blockIdx.x == 0 && threadIdx.x < sizeof(FusedCtl) / 4) reinterpret_cast<unsigned *>(&st->ctl)[threadIdx.x] = 0u;
}

// the one pipeline shape the fused kernel is built for: 16 rows x 3 stages, 8 consumer warps, 2 CTAs per SM
constexpr int kFRows = 16, kFStages = 3, kFWarps = 8, kFMinB = 2;

}  // namespace sx

using namespace sx;

extern "C" size_t sx_fused_state_bytes(void) { return sizeof(FusedState); }
extern "C" size_t sx_fused_state_timestamps_offset(void) { return offsetof(FusedState, ctl) + offsetof(FusedCtl, ts); }

extern "C" int sx_fused_state_init(sx_fused_state *state, int64_t K, void *stream) {
    if (!state || K < 1 || K > SX_TOPK_MAX_K) return SX_ERR_INVALID;
    if (((uintptr_t)state & 15) != 0) return SX_ERR_UNALIGNED;
    fused_init_kernel<<<num_sms(), 256, 0, (cudaStream_t)stream>>>((FusedState *)state, (unsigned)K);
    SX_LAUNCH_CHECK();
    return SX_OK;
}

extern "C" int sx_fused_merge_fits(int64_t K, int G) {
    constexpr size_t ring = (size_t)kFStages * kFRows * kBoxCols * sizeof(double);
    return K >= 1 && G >= 1 && (size_t)K * (size_t)G * 8 <= ring;
}

extern "C" int sx_price_dense_ot_fused(const double *M, int64_t ld, int64_t row0, int64_t S_loc, int64_t D,
                                       const double *y_src, const double *y_dst, double tol,
                                       sx_fused_state *state, double *cand_rc, int64_t *cand_id, int64_t cand_cap,
                                       int64_t K, int64_t *block, int64_t block_len, void *const *peer_bufs_dev,
                                       int rank, int G, int64_t *merged_out, int32_t *status_dev, void *ws,
                                       size_t ws_bytes, void *stream) {
    if (!M || !y_src || !y_dst || !state || !block || S_loc <= 0 || D <= 0 || ld < D || row0 < 0 || cand_cap < 0)
        return SX_ERR_INVALID;
    if (K < 1 || K > SX_TOPK_MAX_K || block_len < 2 * K + 6) return SX_ERR_INVALID;
    if (cand_cap > 0 && (!cand_rc || !cand_id)) return SX_ERR_INVALID;
    if (peer_bufs_dev && (G < 1 || rank < 0 || rank >= G)) return SX_ERR_INVALID;
    if (merged_out && (!peer_bufs_dev || !status_dev)) return SX_ERR_INVALID;
    if (merged_out && !sx_fused_merge_fits(K, G)) return SX_ERR_TOO_LARGE;
    if (!ws || ws_bytes < sx_topk_workspace_bytes(cand_cap, K)) return SX_ERR_WORKSPACE;
    if (((uintptr_t)M % 16) != 0 || (ld % 2) != 0) return SX_ERR_UNALIGNED;
    if (D >= (1ll << 31) || S_loc >= (1ll << 31)) return SX_ERR_TOO_LARGE;
    cudaStream_t st = (cudaStream_t)stream;

    DenseParams p;
    p.y_src = y_src; p.y_dst = y_dst; p.S_loc = S_loc; p.D = D; p.row0 = row0; p.thr = -tol;
    p.sink.hdr = nullptr; p.sink.sel = nullptr;                   // set on the device from the pass parity
    p.sink.rc = cand_rc; p.sink.id = (int64_t *)cand_id; p.sink.cap = cand_cap;
    p.rc_out = nullptr; p.ld_out = 0; p.zero = 0; p.evict_first = 1; p.dyn_ctr = nullptr;
    p.n_col_blocks = (D + kBoxCols - 1) / kBoxCols;
    p.n_row_tiles = (S_loc + kFRows - 1) / kFRows;
    CUtensorMap map;
    int rc = encode_slab_map(&map, M, ld, S_loc, D, kFRows, /*l2_promotion=*/3);
    if (rc != SX_OK) return rc;

    FusedParams f;
    f.state = (FusedState *)state; f.cand_rc = cand_rc; f.cand_id = (const long long *)cand_id; f.cand_cap = cand_cap;
    Carver cv(ws);
    f.K = (unsigned)K; f.block = (long long *)block; f.lists = carve_sel_lists(cv, cand_cap);
    f.peer_bufs = (char *const *)peer_bufs_dev; f.rank = rank; f.G = peer_bufs_dev ? G : 1; f.block_len = block_len;
    f.merged = (long long *)merged_out; f.xstatus = (int *)status_dev; f.timeout_ns = 10ull * 1000 * 1000 * 1000;
    static int steal = -1;
    if (steal < 0) { const char *e = getenv("SX_FUSED_STEAL"); steal = (e && e[0] == '0') ? 0 : 1; }
    f.steal = steal;

    auto kern = price_fused_kernel<kFRows, kFStages, kFWarps, kFMinB>;
    constexpr size_t smem = tma_smem_bytes(kFRows, kFStages, kFWarps);
    constexpr int threads = (kFWarps + 1) * 32;
    static int occ_cached[64] = {0};
    int dev = 0;
    SX_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return SX_ERR_INVALID;
    if (occ_cached[dev] == 0) {
        SX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int occ = 0;
        SX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, smem));
        if (occ < 1) return SX_ERR_NO_DEVICE;
        occ_cached[dev] = occ < kFMinB ? occ : kFMinB;
    }
    const long long total = p.n_row_tiles * p.n_col_blocks;
    long long grid = (long long)num_sms() * occ_cached[dev];
    if (grid > total) grid = total;
    void *args[] = {(void *)&map, (void *)&p, (void *)&f};
    // cooperative: the grid-wide barriers need every CTA resident (a plain launch measured the same speed)
    SX_CUDA(cudaLaunchCooperativeKernel((void *)kern, dim3((unsigned)grid), dim3(threads), args, smem, st));
    return SX_OK;
}

// sx_fused.cu -- one launch per pricing pass: price + select + exchange + merge (sm_100a).
//
// A column-generation pricing pass (reference net_manager.py:474-497, plus the north_star top-k) used to
// be five launches on the critical path -- pass begin (state clear), pricing, cooperative selection, push
// of the result block to the peer GPUs, merge -- and on a row slab of a few hundred MB their launch gaps
// and grid-wide barriers cost as much as the pricing itself.  price_fused_kernel does all of it:
//
//   start    every CTA clears its slice of the OTHER selection state (the pricer owns two, used by
//            alternate passes), so no pass ever waits for a clear;
//   pricing  the TMA pipeline of sx_price_tma.cuh: count, min, candidate list + histogram.  With a lower-bound
//            copy of the slab (sx_cost_lb_build) it streams the copy and re-reads the exact fp64 cost of the
//            few arcs the copy flags; after a dense pass (many violators) it streams M itself;
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
//   merge    the last CTAs of the grid -- which have no rank work -- run merge_ll (sx_merge.cuh), the merge
//            sx_topk_merge_ll runs too: they stage the keys of all G blocks out of the local exchange buffer
//            as they land (staging is the wait), rank every element by G - 1 binary searches in shared
//            memory and write the merged top-K.
//
// If the candidate buffer overflowed, the pass raises SX_STATUS_CAND_OVERFLOW in the header -- it still
// pushes a well-formed block so that no peer waits -- and the caller grows the buffer and repeats the pass.
#include <stdlib.h>
#include <string.h>

#include "sx_gridbar.cuh"
#include "sx_merge.cuh"
#include "sx_price_tma.cuh"

namespace sx {

constexpr int kMergeCtas = 64;          // CTAs (from the end of the grid) that merge the G blocks

struct FusedCtl {
    unsigned long long pass;      // passes completed; parity selects the selection state in use
    GridBarrier        bar;       // grid-wide barrier (sx_gridbar.cuh)
    unsigned int       dyn_ctr;   // tail stealing of the pricing walk: next dynamically assigned tile (0 between passes)
    unsigned int       walk;      // diagnostics: 1 = the last pass streamed the lower-bound copy, 0 = fp64 M
    unsigned long long n_violating_last;   // violators of the last pass on this slab: picks the next pass's walk
    unsigned long long ts[8];     // diagnostics: %globaltimer of CTA 0 at the phase boundaries of the last pass
};
// Pricer.fused_walk reads `walk` 12 bytes before the timestamps
static_assert(offsetof(FusedCtl, ts) - offsetof(FusedCtl, walk) == 12, "");
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
    int              has_lb;         // 1: the lower-bound copy is there (second tensor map)
    unsigned long long lb_max_violating;   // walk the copy while the last pass had at most this many violators
};

__device__ __forceinline__ unsigned long long ld_volatile_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void stamp(FusedCtl *ctl, int i) {
    if (blockIdx.x == 0 && threadIdx.x == 0) ctl->ts[i] = global_timer_ns();
}

// 2 CTAs per SM hold at most 96 registers per thread: the 18 warps land 5 / 5 / 4 / 4 on the SM's four
// sub-partitions, whose register files hold 16 384 registers each (112 per thread would pass a whole-SM count
// but leave one CTA per SM).
// EXT_IDS: arc ids in the big-M extension's numbering (p.id_ld = D + 1; see price_tiles).
template <int ROWS, int STAGES, int LB_STAGES, int CWARPS, int MINB, bool EXT_IDS>
__global__ void __launch_bounds__((CWARPS + 1) * 32, MINB)
price_fused_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap tmap_lb,
                   const DenseParams p0, const FusedParams f) {
    static_assert((size_t)STAGES * ROWS * kBoxCols * sizeof(double) >= sizeof(SelScratch),
                  "the stage ring is reused as the selection's shared memory");
    static_assert((size_t)LB_STAGES * ROWS * kBoxCols * sizeof(uint32_t) == (size_t)STAGES * ROWS * kBoxCols * sizeof(double),
                  "both walks use the same ring (the barriers follow it)");
    static_assert(CWARPS * 32 == kSelThreads, "the consumer warps select, the producer warp joins the barriers");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ MergeFold s_fold;
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
        ll_ctr = ll_counters(ll_local, f.G, f.block_len);
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
    // The walk of this pass: the lower-bound copy (4 B per arc, flagged arcs re-read from M) unless the last
    // pass on this state was dense, where the re-reads would cost more than the fp64 walk (DESIGN.md 5).
    // n_violating_last is written after barrier 1 of a pass, so every CTA reads the same value here.
    const bool lb_walk = f.has_lb && ld_volatile_u64(&ctl->n_violating_last) <= f.lb_max_violating;
    if (lb_walk) price_tiles<uint32_t, ROWS, LB_STAGES, CWARPS, false, EXT_IDS>(tmap_lb, p, smem_raw);
    else         price_tiles<double, ROWS, STAGES, CWARPS, false, EXT_IDS>(tmap, p, smem_raw);
    if (blockIdx.x == 0 && tid == 0) ctl->walk = lb_walk ? 1u : 0u;
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
                    ll_store_slot(ll_slot(f.peer_bufs[q], f.G, f.block_len, epoch, f.rank, rank), flag, rc_bits);
                    ll_store_slot(ll_slot(f.peer_bufs[q], f.G, f.block_len, epoch, f.rank, (long long)K + rank), flag,
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
                    ll_store_slot(ll_slot(f.peer_bufs[q], f.G, f.block_len, epoch, f.rank, i), flag, pad_rc);
                    ll_store_slot(ll_slot(f.peer_bufs[q], f.G, f.block_len, epoch, f.rank, (long long)K + i), flag, ~0ull);
                }
        }
        if (tid < 6) {
            unsigned long long w = 0;
            if (tid == 0) { w = __ldcg(&sel->hdr.n_violating); ctl->n_violating_last = w; }
            if (tid == 1) w = (unsigned long long)__ldcg(&sel->hdr.min_rc_key);
            if (tid == 2) w = __ldcg(&sel->hdr.n_priced);
            if (tid == 3)
                w = __ldcg(&sel->hdr.status) | (n64 > (unsigned long long)f.cand_cap ? kStatusCandOverflow : 0ull) |
                    (sr.duplicates ? kStatusDuplicateCandidates : 0ull);
            if (tid == 4) w = (unsigned long long)n_out;
            f.block[2 * K + tid] = (long long)w;
            if (f.peer_bufs)
                for (int q = 0; q < f.G; ++q)
                    ll_store_slot(ll_slot(f.peer_bufs[q], f.G, f.block_len, epoch, f.rank, (long long)2 * K + tid), flag, w);
        }
    }

    if (blockIdx.x == gridDim.x - 1 && tid == 0) ctl->ts[6] = global_timer_ns();   // overwritten at the end of the merge
    // ---- merge of the G blocks out of the local exchange buffer (merge_ll, sx_merge.cuh) ----
    if (f.peer_bufs == nullptr || f.merged == nullptr) return;
    const int n_merge = gridDim.x < kMergeCtas ? (int)gridDim.x : kMergeCtas;
    const int mc = (int)blockIdx.x - ((int)gridDim.x - n_merge);           // index among the merge CTAs
    if (mc < 0) return;
    // the stage ring holds the G * K keys: the rank tiles are no longer read
    if (!merge_ll(ll_local, f.block_len, f.G, K, epoch, mc, n_merge, reinterpret_cast<unsigned long long *>(smem_raw),
                  s_fold, f.merged, f.merged + K, f.merged + 2 * K, f.merged + 2 * K + 1, f.timeout_ns))
        atomicExch(f.xstatus, SX_ERR_PEER_TIMEOUT);
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

// The border of the big-M extension (reference net_manager.py:390-393) of one row shard, priced into the selection
// state the NEXT price_fused_kernel launch on this stream uses: arcs (i, D) at cost bigM for the shard's rows and,
// on the shard that ends at S, the artificial row (S, j) at cost bigM and the corner (S, D) at cost `corner`.  The
// fused kernel then prices the base slab with arc ids i (D + 1) + j (p.id_ld = D + 1), so count, minimum, NaN status
// and candidates are those of the physically extended (S + 1) x (D + 1) matrix, without a copy of it.
//
// Why sel[ctl.pass & 1] is the right state, and clear: a fused pass reads `pass` at its start, prices into that
// half, clears the OTHER half at its start and advances `pass` after barrier 1; sx_fused_state_init clears both
// halves before the first pass.  So once the previous launch on the stream has finished, sel[pass & 1] is clear
// and is the one the next fused launch prices into -- this kernel runs between the two.  It takes the violator
// path of the walk (tile_epilogue / WarpTally / block_min_commit): exact count and minimum, NaN reduced costs raise
// SX_STATUS_NAN_RC without being counted or selected, candidates are appended under the histogram bound.
__global__ void __launch_bounds__(256) price_border_kernel(const DenseParams p0, FusedState *state,
                                                          const double *y_art, long long S, double bigM,
                                                          double corner) {
    __shared__ long long scratch[256 / 32];
    SelState *sel = &state->sel[ld_volatile_u64(&state->ctl.pass) & 1ull];
    DenseParams p = p0;
    p.sink.hdr = &sel->hdr;
    p.sink.sel = sel;
    const long long n_col = p.S_loc;                                     // (row0 + i, D), i < S_loc
    const long long n = n_col + (p.row0 + p.S_loc == S ? p.D + 1 : 0);   // + (S, j), j <= D
    const double v_art = __ldg(p.y_dst + p.D);
    double tmin = INFINITY, lim = INFINITY;
    WarpTally tally;
    // the loop bound is uniform per block: every lane of a warp joins the votes of tile_epilogue
    for (long long base = (long long)blockIdx.x * blockDim.x; base < n; base += (long long)gridDim.x * blockDim.x) {
        const long long k = base + threadIdx.x;
        double rc0[1] = {INFINITY}, rc1[1] = {INFINITY};
        long long id = 0;
        if (k < n_col) {
            rc0[0] = bigM - (v_art - __ldg(p.y_src + k));
            id = (p.row0 + k) * p.id_ld + p.D;
        } else if (k < n) {
            const long long j = k - n_col;
            rc0[0] = (j < p.D ? bigM : corner) - (__ldg(p.y_dst + j) - __ldg(y_art));
            id = S * p.id_ld + j;
        }
        tile_epilogue<1>(p, tally, tmin, lim, rc0, rc1, lt_or(rc0[0], lim, false), id, 0);
    }
    warp_flush(p.sink, tally);
    block_min_commit(tmin, p.sink.hdr, scratch, 256 / 32, threadIdx.x >> 5, (unsigned long long)n);
}

struct BigMBorder {
    long long     S;        // rows of the base matrix; the artificial row is S
    const double *y_art;    // device: u_S
    double        bigM, corner;
};

// the one pipeline shape the fused kernel is built for: 16 rows x 3 stages (fp64; 6 stages of the 4-byte copy: the
// same 96 KB ring), 8 consumer warps, 2 CTAs per SM
constexpr int kFRows = 16, kFStages = 3, kFLbStages = 6, kFWarps = 8, kFMinB = 2;

// The lower-bound walk is chosen while the last pass had at most this fraction of the slab's arcs violating.
// Measured at 20 000^2 on a B200 (DESIGN.md 5): the copy walk takes 0.37 / 0.42 / 0.57 / 1.07 ms at 1e-5 /
// 1e-4 / 1e-3 / 1e-2 violating, the fp64 walk 0.46 / 0.46 / 0.48 / 0.64 ms: they cross near 5e-4.
// SX_FUSED_LB_MAX_FRAC overrides it (to measure the crossover).
constexpr double kLbMaxViolatingFrac = 1.0 / 2048;

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
    return sx_price_dense_ot_fused_lb(M, ld, nullptr, 0, row0, S_loc, D, y_src, y_dst, tol, state, cand_rc, cand_id,
                                      cand_cap, K, block, block_len, peer_bufs_dev, rank, G, merged_out, status_dev, ws,
                                      ws_bytes, stream);
}

namespace {

// The fused pass over a base slab; with `bm` the border kernel first prices the big-M border into the same pass and
// arc ids take the extended row stride D + 1.  Every argument is checked and both tensor maps are encoded before
// the first launch, so a rejected call launches nothing.
int fused_pass(const double *M, int64_t ld, const uint32_t *lb, int64_t ld_lb, int64_t row0, int64_t S_loc, int64_t D,
               const double *y_src, const double *y_dst, double tol, sx_fused_state *state, double *cand_rc,
               int64_t *cand_id, int64_t cand_cap, int64_t K, int64_t *block, int64_t block_len,
               void *const *peer_bufs_dev, int rank, int G, int64_t *merged_out, int32_t *status_dev, void *ws,
               size_t ws_bytes, void *stream, const BigMBorder *bm) {
    if (!M || !y_src || !y_dst || !state || !block || S_loc <= 0 || D <= 0 || ld < D || row0 < 0 || cand_cap < 0)
        return SX_ERR_INVALID;
    if (K < 1 || K > SX_TOPK_MAX_K || block_len < 2 * K + 6) return SX_ERR_INVALID;
    if (cand_cap > 0 && (!cand_rc || !cand_id)) return SX_ERR_INVALID;
    if (peer_bufs_dev && (G < 1 || rank < 0 || rank >= G)) return SX_ERR_INVALID;
    if (merged_out && (!peer_bufs_dev || !status_dev)) return SX_ERR_INVALID;
    if (merged_out && !sx_fused_merge_fits(K, G)) return SX_ERR_TOO_LARGE;
    if (!ws || ws_bytes < sx_topk_workspace_bytes(cand_cap, K)) return SX_ERR_WORKSPACE;
    if (((uintptr_t)M % 16) != 0 || (ld % 2) != 0) return SX_ERR_UNALIGNED;
    if (lb && ld_lb < D) return SX_ERR_INVALID;
    if (lb && (((uintptr_t)lb % 16) != 0 || (ld_lb % 4) != 0)) return SX_ERR_UNALIGNED;   // 16 B TMA row stride
    if (D >= (1ll << 31) || S_loc >= (1ll << 31)) return SX_ERR_TOO_LARGE;
    cudaStream_t st = (cudaStream_t)stream;

    DenseParams p;
    p.y_src = y_src; p.y_dst = y_dst; p.M = M; p.ld = ld; p.S_loc = S_loc; p.D = D; p.row0 = row0;
    p.id_ld = bm ? D + 1 : D; p.thr = -tol;
    p.sink.hdr = nullptr; p.sink.sel = nullptr;                   // set on the device from the pass parity
    p.sink.rc = cand_rc; p.sink.id = (int64_t *)cand_id; p.sink.cap = cand_cap;
    p.rc_out = nullptr; p.ld_out = 0; p.zero = 0; p.evict_first = 1; p.dyn_ctr = nullptr;
    p.n_col_blocks = (D + kBoxCols - 1) / kBoxCols;
    p.n_row_tiles = (S_loc + kFRows - 1) / kFRows;
    CUtensorMap map, map_lb;
    int rc = encode_slab_map(&map, M, ld, S_loc, D, kFRows, /*l2_promotion=*/3);
    if (rc != SX_OK) return rc;
    memset(&map_lb, 0, sizeof(map_lb));
    if (lb && (rc = encode_slab_map(&map_lb, lb, ld_lb, S_loc, D, kFRows, /*l2_promotion=*/3)) != SX_OK) return rc;

    FusedParams f;
    f.state = (FusedState *)state; f.cand_rc = cand_rc; f.cand_id = (const long long *)cand_id; f.cand_cap = cand_cap;
    Carver cv(ws);
    f.K = (unsigned)K; f.block = (long long *)block; f.lists = carve_sel_lists(cv, cand_cap);
    f.peer_bufs = (char *const *)peer_bufs_dev; f.rank = rank; f.G = peer_bufs_dev ? G : 1; f.block_len = block_len;
    f.merged = (long long *)merged_out; f.xstatus = (int *)status_dev; f.timeout_ns = 10ull * 1000 * 1000 * 1000;
    static int steal = -1;
    if (steal < 0) { const char *e = getenv("SX_FUSED_STEAL"); steal = (e && e[0] == '0') ? 0 : 1; }
    f.steal = steal;
    static double lb_frac = -1.0;
    if (lb_frac < 0) { const char *e = getenv("SX_FUSED_LB_MAX_FRAC"); lb_frac = e ? atof(e) : kLbMaxViolatingFrac; }
    f.has_lb = lb ? 1 : 0;
    f.lb_max_violating = (unsigned long long)(lb_frac * (double)S_loc * (double)D);

    auto kern = bm ? price_fused_kernel<kFRows, kFStages, kFLbStages, kFWarps, kFMinB, true>
                   : price_fused_kernel<kFRows, kFStages, kFLbStages, kFWarps, kFMinB, false>;
    constexpr size_t smem_f64 = tma_smem_bytes(kFRows, kFStages, kFWarps),
                     smem_lb = tma_smem_bytes(kFRows, kFLbStages, kFWarps, sizeof(uint32_t));
    constexpr size_t smem = smem_f64 > smem_lb ? smem_f64 : smem_lb;
    constexpr int threads = (kFWarps + 1) * 32;
    static int occ_cache[2][64] = {{0}};
    int *occ_cached = occ_cache[bm ? 1 : 0];
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
    if (bm) {
        const long long n = S_loc + (row0 + S_loc == bm->S ? D + 1 : 0);
        long long bgrid = (n + 255) / 256;
        if (bgrid > (long long)num_sms() * 4) bgrid = (long long)num_sms() * 4;
        price_border_kernel<<<(unsigned)bgrid, 256, 0, st>>>(p, f.state, bm->y_art, bm->S, bm->bigM, bm->corner);
        SX_LAUNCH_CHECK();
    }
    void *args[] = {(void *)&map, (void *)&map_lb, (void *)&p, (void *)&f};
    // cooperative: the grid-wide barriers need every CTA resident (a plain launch measured the same speed)
    SX_CUDA(cudaLaunchCooperativeKernel((void *)kern, dim3((unsigned)grid), dim3(threads), args, smem, st));
    return SX_OK;
}

}  // namespace

extern "C" int sx_price_dense_ot_fused_lb(const double *M, int64_t ld, const uint32_t *lb, int64_t ld_lb, int64_t row0,
                                          int64_t S_loc, int64_t D, const double *y_src, const double *y_dst,
                                          double tol, sx_fused_state *state, double *cand_rc, int64_t *cand_id,
                                          int64_t cand_cap, int64_t K, int64_t *block, int64_t block_len,
                                          void *const *peer_bufs_dev, int rank, int G, int64_t *merged_out,
                                          int32_t *status_dev, void *ws, size_t ws_bytes, void *stream) {
    return fused_pass(M, ld, lb, ld_lb, row0, S_loc, D, y_src, y_dst, tol, state, cand_rc, cand_id, cand_cap, K, block,
                      block_len, peer_bufs_dev, rank, G, merged_out, status_dev, ws, ws_bytes, stream, nullptr);
}

extern "C" int sx_price_dense_ot_fused_bigm(const double *M, int64_t ld, const uint32_t *lb, int64_t ld_lb,
                                            int64_t row0, int64_t S_loc, int64_t S, int64_t D, const double *y_src,
                                            const double *y_dst, const double *y_art, double bigM, double corner,
                                            double tol, sx_fused_state *state, double *cand_rc, int64_t *cand_id,
                                            int64_t cand_cap, int64_t K, int64_t *block, int64_t block_len,
                                            void *const *peer_bufs_dev, int rank, int G, int64_t *merged_out,
                                            int32_t *status_dev, void *ws, size_t ws_bytes, void *stream) {
    if (S_loc <= 0 || row0 < 0 || S < 1 || row0 + S_loc > S) return SX_ERR_INVALID;
    if (row0 + S_loc == S && !y_art) return SX_ERR_INVALID;
    if (D + 1 >= (1ll << 31)) return SX_ERR_TOO_LARGE;
    const BigMBorder bm{S, y_art, bigM, corner};
    return fused_pass(M, ld, lb, ld_lb, row0, S_loc, D, y_src, y_dst, tol, state, cand_rc, cand_id, cand_cap, K, block,
                      block_len, peer_bufs_dev, rank, G, merged_out, status_dev, ws, ws_bytes, stream, &bm);
}

// sx_price_tma.cuh -- the TMA-staged dense pricing pass of one CTA (sm_100a) and what it needs: mbarrier /
// cp.async.bulk.tensor PTX wrappers, the violator accounting shared by all pricing kernels, the tensor-map
// encoder.  Included by sx_price.cu (price_dense_tma_kernel) and sx_fused.cu (price + select + push in one
// launch).  See sx_price.cu for the description of the pass.
#pragma once
#include <cuda.h>
#include <math.h>

#include <type_traits>

#include "sx_common.cuh"
#include "sx_select.cuh"

namespace sx {

// ---------------------------------------------------------------------------------------
// PTX helpers: mbarrier + TMA (cp.async.bulk.tensor)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
// Arrive that cannot be issued before `dep` is known.  A consumer releases a stage once its data
// is in registers; "the loads were issued" is not enough (an LDS queued behind global atomics can
// still be in flight when the arrive lets the producer's TMA overwrite the stage), so the release
// carries a register dependency on a value computed from every loaded element.
// `dep_times_zero` = dep * (a zero only known at run time): folded into the barrier address.
__device__ __forceinline__ void mbar_arrive_after(uint64_t *bar, uint32_t dep_times_zero) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar) + dep_times_zero) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra.uni WAIT_DONE;\n"
        "bra.uni WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint64_t l2_evict_normal_policy() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void tma_load_2d(void *smem_dst, const CUtensorMap *map, uint64_t *bar,
                                            int c0, int c1, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(smem_u32(smem_dst)),
        "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "l"(policy)
        : "memory");
}

// acc || !(a >= b) as ONE predicated compare (setp.ltu.or.f64: "less than or unordered").  Written in PTX
// because the compiler otherwise rewrites an OR of "x_i < lim" into "min(x_i) < lim", and an fp64 min is
// ~8 instructions.  Unordered on purpose: a NaN reduced cost must reach the epilogue, where it raises
// SX_STATUS_NAN_RC -- the reference's `np.all(rc >= -tol)` (net_manager.py:496) is False for it.
__device__ __forceinline__ bool lt_or(double a, double b, bool acc) {
    int r;
    asm("{\n"
        ".reg .pred p, q;\n"
        "setp.ne.s32 q, %3, 0;\n"
        "setp.ltu.or.f64 p, %1, %2, q;\n"
        "selp.s32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(r)
        : "d"(a), "d"(b), "r"((int)acc));
    return r != 0;
}

// ---------------------------------------------------------------------------------------
// Violator accounting shared by all pricing kernels (rare path: a tile with at least one
// violator).  Violators are COUNTED exactly in a per-warp register (one atomicAdd per warp at
// kernel end); they are APPENDED to the candidate list only while they can still be among the
// K most violating arcs, i.e. while their histogram bin is <= SelState::bstar (sx_select.cuh).
// ---------------------------------------------------------------------------------------
struct CandSink {
    sx_price_header *hdr;
    SelState        *sel;   // nullptr <=> cap == 0 (count / min only)
    double          *rc;
    int64_t         *id;
    long long        cap;
};

struct WarpTally {
    unsigned long long count = 0;   // violators seen by this warp (same value in every lane)
};

// NE elements per thread, given by val(e) / id(e) with e a compile-time index after unrolling.
template <int NE, class ValFn, class IdFn>
__device__ __forceinline__ void emit_violators(const CandSink &sink, WarpTally &tally, double thr, ValFn val,
                                               IdFn id) {
    unsigned nviol = 0;
#pragma unroll
    for (int e = 0; e < NE; ++e) nviol += __popc(__ballot_sync(0xffffffffu, val(e) < thr));
    tally.count += nviol;
    if (sink.cap == 0 || nviol == 0) return;
    SelState *st = sink.sel;
    unsigned bs = 0;
    if (lane_id() == 0) bs = ld_relaxed_u32(&st->bstar);
    bs = __shfl_sync(0xffffffffu, bs, 0);
    unsigned qm = 0;
#pragma unroll
    for (int e = 0; e < NE; ++e) {
        const double v = val(e);
        if (v < thr && cand_bin(v) <= bs) qm |= 1u << e;
    }
    const unsigned mine = __popc(qm);
    unsigned incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane_id() >= o) incl += t;
    }
    const unsigned total = __shfl_sync(0xffffffffu, incl, 31);
    if (total == 0) return;
    unsigned long long base = 0;
    if (lane_id() == 0) base = atomicAdd(&st->n_cand, (unsigned long long)total);
    base = __shfl_sync(0xffffffffu, base, 0);
    long long slot = (long long)base + (incl - mine);
    bool dropped = false;
#pragma unroll
    for (int e = 0; e < NE; ++e) {
        if (qm & (1u << e)) {
            const double v = val(e);
            if (slot < sink.cap) { sink.rc[slot] = v; sink.id[slot] = id(e); } else dropped = true;
            ++slot;
            atomicAdd(&st->fine[cand_bin(v)], 1u);
        }
    }
    if (dropped) atomicOr(&sink.hdr->status, kStatusCandOverflow);
    __threadfence();   // fine before top: the coarse level never runs ahead of the fine one
#pragma unroll
    for (int e = 0; e < NE; ++e)
        if (qm & (1u << e)) atomicAdd(&st->top[cand_bin(val(e)) >> 8], 1u);
    // every kTightenPeriod candidates the warp that crosses the mark lowers the bound
    const unsigned long long after = base + total;
    if (base / kTightenPeriod != after / kTightenPeriod && after >= st->K) {
        const unsigned b = warp_find_bound(st, st->K, nullptr);
        if (lane_id() == 0 && b < bs) atomicMin(&st->bstar, b);
    }
}
__device__ __forceinline__ void warp_flush(const CandSink &sink, const WarpTally &tally) {
    if (lane_id() == 0 && tally.count) atomicAdd(&sink.hdr->n_violating, tally.count);
}

// Block-level min -> one atomicMin per CTA.
__device__ __forceinline__ void block_min_commit(double tmin, sx_price_header *hdr, long long *smem_scratch,
                                                 int n_warps, int warp, unsigned long long n_priced) {
    long long k = f64_to_min_key(tmin);
    k = warp_min(k);
    if (lane_id() == 0) smem_scratch[warp] = k;
    __syncthreads();
    if (threadIdx.x == 0) {
        long long m = smem_scratch[0];
        for (int w = 1; w < n_warps; ++w) m = smem_scratch[w] < m ? smem_scratch[w] : m;
        atomicMin(&hdr->min_rc_key, m);
        if (blockIdx.x == 0) atomicAdd(&hdr->n_priced, n_priced);
    }
}

// ---------------------------------------------------------------------------------------
// K4a, variant 0: TMA pipeline
// ---------------------------------------------------------------------------------------
constexpr int kBoxCols = 256;   // elements per box row (TMA max box dim)

struct DenseParams {
    const double *y_src;   // S_loc
    const double *y_dst;   // D
    const double *M;       // the slab itself: the lower-bound walk re-reads flagged arcs from it
    long long     ld;
    long long     S_loc, D, row0;
    double        thr;     // -tol
    CandSink      sink;
    double       *rc_out;  // optional
    long long     ld_out;
    long long     n_col_blocks, n_row_tiles;
    uint32_t      zero;    // 0, but only the host knows: see mbar_arrive_after
    uint32_t      evict_first;
    unsigned int *dyn_ctr; // tail stealing: device counter (0 at kernel start) or nullptr = static walk only
    long long     id_ld;   // row stride of arc ids: D, or D + 1 when the slab is priced as part of a big-M extension
};

// Lazy epilogue of one warp's share of a tile: RPT rows x 2 columns per thread already in registers
// as reduced costs (+inf where masked).  The hot loop does ONE compare per reduced cost, against
// lim = max(running min, -tol): a hit means "new minimum or violator", both rare, and only then are
// the exact minimum updated and the violators counted / appended (fp64 min costs ~8 SASS
// instructions on sm_100a).
template <int RPT>
__device__ __forceinline__ void tile_epilogue(const DenseParams &p, WarpTally &tally, double &tmin, double &lim,
                                              const double (&rc0)[RPT], const double (&rc1)[RPT], bool hit,
                                              long long gid0, long long row_stride, int col_gap = 1) {
    if (!__any_sync(0xffffffffu, hit)) return;
    bool viol = false;
    if (hit) {
        double mn = tmin;
        bool nan = false;
#pragma unroll
        for (int r = 0; r < RPT; ++r) {
            mn = rc0[r] < mn ? rc0[r] : mn;
            mn = rc1[r] < mn ? rc1[r] : mn;
            viol = viol || (rc0[r] < p.thr) || (rc1[r] < p.thr);
            nan = nan || (rc0[r] != rc0[r]) || (rc1[r] != rc1[r]);
        }
        tmin = mn;
        lim = tmin > p.thr ? tmin : p.thr;
        if (nan) atomicOr(&p.sink.hdr->status, kStatusNanRc);
    }
    if (__any_sync(0xffffffffu, viol))
        emit_violators<2 * RPT>(
            p.sink, tally, p.thr, [&](int e) { return (e & 1) ? rc1[e >> 1] : rc0[e >> 1]; },
            [&](int e) { return gid0 + (long long)(e >> 1) * row_stride + ((e & 1) ? col_gap : 0); });
}

// CWARPS consumer warps: 4 warps span the 256 box columns (2 adjacent columns per thread, so a
// warp reads 512 (fp64) / 256 (fp32) contiguous bytes of a box row: conflict-free), CWARPS/4 row groups.
// The whole pricing pass of one CTA as a device function (shared by price_dense_tma_kernel and the fused
// price + select + push kernel, sx_fused.cu).  Returns after a __syncthreads(): every TMA load of this CTA
// has been consumed, so the caller may reuse the shared memory.
//
// T = double: the map streams M itself (8 B per arc).
// T = uint32_t: the map streams the lower-bound copy (sx_cost_lb_build, 4 B per arc): the high word of each
//   fp64 cost rounded toward -inf, so L = that word as the high half of a double (low half 0) -- a register
//   move, not a conversion -- and M is re-read from global memory only for the arcs L flags.  Why that is
//   exact: L <= M elementwise (or L is NaN), and fp64 subtraction of the same w = fl(v - u) is monotone, so
//   rc_lb = fl(L - w) <= fl(M - w) = rc.  The filter flags an arc when !(rc_lb >= lim), lim = max(running min, -tol); an arc it does not
//   flag has rc >= rc_lb >= lim, so it is neither a violator (rc >= -tol) nor below the running minimum,
//   and it is not NaN (a NaN rc needs M or w NaN, or M and w infinite of one sign -- L keeps NaN and
//   infinities, so rc_lb is NaN then too).  Flagged arcs get rc = M - (v - u) from the exact M, the same
//   operations as the fp64 walk, and unflagged ones enter the epilogue as +inf.  The running minimum is
//   only ever updated from exact values, so count, minimum, NaN status and candidates are those of the
//   fp64 walk, bit for bit.
//
// EXT_IDS: arc ids take the row stride p.id_ld (the big-M extension's D + 1) instead of p.D.  A compile-time choice:
// a second loop-invariant stride live across the walk changes the register allocation (and the spills) of the
// kernels that never need it, and every kernel built before the extension sets id_ld = D anyway.
template <class T, int ROWS, int STAGES, int CWARPS, bool WRITE_RC, bool EXT_IDS = false>
__device__ __forceinline__ void price_tiles(const CUtensorMap &tmap, const DenseParams &p, unsigned char *smem_raw) {
    static_assert(sizeof(T) == 8 || !WRITE_RC, "the lower-bound walk does not write reduced costs");
    static_assert(std::is_same<T, double>::value || std::is_same<T, uint32_t>::value, "fp64 M or its lower-bound words");
    using T2 = typename std::conditional<sizeof(T) == 8, double2, uint2>::type;
    constexpr int      RPT         = ROWS / (CWARPS / 4);      // rows per consumer thread
    constexpr uint32_t kStageBytes = ROWS * kBoxCols * sizeof(T);
    T        *stage_base = reinterpret_cast<T *>(smem_raw);
    uint64_t *full_bar   = reinterpret_cast<uint64_t *>(smem_raw + (size_t)STAGES * kStageBytes);
    uint64_t *empty_bar  = full_bar + STAGES;
    long long *scratch   = reinterpret_cast<long long *>(empty_bar + STAGES);

    const int warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], CWARPS);
        }
        mbar_fence_init();
    }
    __syncthreads();

    // Grid-stride tile walk, tile t = row_tile * n_col_blocks + col_block: at any time the CTAs of
    // the grid read neighbouring 2 KB segments of the same few matrix rows (DRAM page locality).
    // With p.dyn_ctr the last eighth of the tiles is not assigned up front but handed out by an atomic
    // counter ("tail stealing"): SMs stream at visibly different rates (the slowest CTA of a static walk
    // finishes 3-7 % after the fastest, and everybody waits for it at the grid barrier that follows), so
    // the fast ones take more of the tail.  The producer publishes each dynamic tile's index in shared
    // memory before it arms the stage's barrier; consumers read it after the barrier's wait.
    const long long total = p.n_row_tiles * p.n_col_blocks;
    const long long G = gridDim.x;
    long long rt = (long long)blockIdx.x / p.n_col_blocks;
    long long cb = (long long)blockIdx.x - rt * p.n_col_blocks;
    const long long d_rt = G / p.n_col_blocks, d_cb = G - d_rt * p.n_col_blocks;
    const bool dynamic = p.dyn_ctr != nullptr;
    // static tiles of this CTA: all of its grid-stride share, or 7/8 of the common share when the tail is dynamic
    const long long share = total / G;
    const long long n_static = dynamic ? share - share / 8 : (total - (long long)blockIdx.x + G - 1) / G;
    const long long dyn_base = n_static * G;                                 // first dynamically assigned tile
    volatile long long *ticket = reinterpret_cast<volatile long long *>(scratch + CWARPS);

    if (warp == CWARPS) {
        // ===== producer warp: one elected lane issues the TMA loads =====
        if (lane_id() == 0) {
            const uint64_t pol = p.evict_first ? l2_evict_first_policy() : l2_evict_normal_policy();
            uint32_t it = 0;
            for (long long k = 0; k < n_static; ++k, ++it) {
                const int s = it % STAGES;
                if (it >= STAGES) mbar_wait(&empty_bar[s], ((it / STAGES) - 1) & 1);
                mbar_arrive_expect_tx(&full_bar[s], kStageBytes);
                tma_load_2d(stage_base + (size_t)s * ROWS * kBoxCols, &tmap, &full_bar[s],
                            (int)(cb * kBoxCols), (int)(rt * ROWS), pol);
                rt += d_rt; cb += d_cb;
                if (cb >= p.n_col_blocks) { cb -= p.n_col_blocks; ++rt; }
            }
            if (dynamic) {
                long long t_next = dyn_base + (long long)atomicAdd(p.dyn_ctr, 1u);
                for (;; ++it) {
                    const int s = it % STAGES;
                    const long long t = t_next;
                    if (t < total) t_next = dyn_base + (long long)atomicAdd(p.dyn_ctr, 1u);   // in flight during the waits
                    if (it >= STAGES) mbar_wait(&empty_bar[s], ((it / STAGES) - 1) & 1);
                    ticket[s] = t < total ? t : -1;
                    if (t >= total) { mbar_arrive_after(&full_bar[s], 0u); break; }          // sentinel: no data follows
                    const long long trt = t / p.n_col_blocks, tcb = t - trt * p.n_col_blocks;
                    mbar_arrive_expect_tx(&full_bar[s], kStageBytes);
                    tma_load_2d(stage_base + (size_t)s * ROWS * kBoxCols, &tmap, &full_bar[s],
                                (int)(tcb * kBoxCols), (int)(trt * ROWS), pol);
                }
            }
        }
    } else {
        // ===== consumer warps =====
        const int c  = threadIdx.x & 127;            // column pair inside the box
        const int rg = threadIdx.x >> 7;             // row group
        double    tmin = INFINITY, lim = INFINITY;
        WarpTally tally;
        // one tile: (rt, cb) in stage s of pipeline iteration it; `waited` = the stage's data is known to be there
        auto process = [&](long long rt, long long cb, int s, uint32_t it, bool waited) {
            const long long id_ld = EXT_IDS ? p.id_ld : p.D;
            const long long j0 = cb * kBoxCols + 2 * c;
            const long long i0 = rt * ROWS + (long long)rg * RPT;
            const bool interior = (cb + 1) * kBoxCols <= p.D && (rt + 1) * ROWS <= p.S_loc;   // CTA-uniform
            // potentials of this thread's columns / rows: issued before the wait so their latency
            // hides behind the TMA transfer
            double v0, v1, u[RPT];
            if (interior) {
                const double2 vv = make_double2(__ldg(p.y_dst + j0), __ldg(p.y_dst + j0 + 1));
                v0 = vv.x; v1 = vv.y;
#pragma unroll
                for (int r = 0; r < RPT; ++r) u[r] = __ldg(p.y_src + i0 + r);
            } else {
                v0 = (j0 < p.D) ? __ldg(p.y_dst + j0) : 0.0;
                v1 = (j0 + 1 < p.D) ? __ldg(p.y_dst + j0 + 1) : 0.0;
#pragma unroll
                for (int r = 0; r < RPT; ++r) u[r] = (i0 + r < p.S_loc) ? __ldg(p.y_src + i0 + r) : 0.0;
            }
            if (!waited) mbar_wait(&full_bar[s], (it / STAGES) & 1);
            const T2 *tile = reinterpret_cast<const T2 *>(stage_base + (size_t)s * ROWS * kBoxCols) +
                             (size_t)rg * RPT * (kBoxCols / 2) + c;
            T2 m[RPT];
#pragma unroll
            for (int r = 0; r < RPT; ++r) m[r] = tile[(size_t)r * (kBoxCols / 2)];
            // Release the slot once the data has ARRIVED in registers: the vote below cannot issue before
            // every lane's shared loads have completed (it consumes one word of each), and the arrive's
            // address depends on the vote.
            uint32_t landed = 0;
#pragma unroll
            for (int r = 0; r < RPT; ++r) {
                if constexpr (sizeof(T) == 8) landed ^= (uint32_t)__double2loint(m[r].x);
                else landed ^= m[r].x;
            }
            const bool rel = __any_sync(0xffffffffu, landed == 0x5a5a5a5au);
            if (lane_id() == 0) mbar_arrive_after(&empty_bar[s], (uint32_t)rel * p.zero);

            if constexpr (sizeof(T) == 4) {
                // lower-bound filter: two fp64 subtractions and one compare per arc, as the fp64 walk
                auto L = [](uint32_t w) { return __hiloint2double((int)w, 0); };
                const bool ok0 = j0 < p.D, ok1 = j0 + 1 < p.D;
                bool hit = false;
                if (interior) {
#pragma unroll
                    for (int r = 0; r < RPT; ++r)
                        hit = lt_or(L(m[r].y) - (v1 - u[r]), lim, lt_or(L(m[r].x) - (v0 - u[r]), lim, hit));
                } else {
#pragma unroll
                    for (int r = 0; r < RPT; ++r) {
                        const bool rok = i0 + r < p.S_loc;
                        const bool f0 = lt_or(L(m[r].x) - (v0 - u[r]), lim, false);
                        const bool f1 = lt_or(L(m[r].y) - (v1 - u[r]), lim, false);
                        hit = hit || (rok && ((f0 && ok0) || (f1 && ok1)));
                    }
                }
                if (!__any_sync(0xffffffffu, hit)) return;
                // rare path: the exact fp64 M of the flagged arcs, the reduced costs rebuilt as the fp64 walk
                // builds them, +inf for the others
                double rc0[RPT], rc1[RPT];
                const double *row = p.M + i0 * p.ld + j0;
#pragma unroll
                for (int r = 0; r < RPT; ++r) {
                    const bool rok = interior || i0 + r < p.S_loc;
                    const double w0 = v0 - u[r], w1 = v1 - u[r];
                    const bool f0 = rok && (interior || ok0) && lt_or(L(m[r].x) - w0, lim, false);
                    const bool f1 = rok && (interior || ok1) && lt_or(L(m[r].y) - w1, lim, false);
                    rc0[r] = f0 ? __ldg(row + (long long)r * p.ld) - w0 : INFINITY;
                    rc1[r] = f1 ? __ldg(row + (long long)r * p.ld + 1) - w1 : INFINITY;
                }
                tile_epilogue<RPT>(p, tally, tmin, lim, rc0, rc1, hit, (p.row0 + i0) * id_ld + j0, id_ld);
                return;
            }
            double rc0[RPT], rc1[RPT];
            bool   hit = false;
            if (interior) {
#pragma unroll
                for (int r = 0; r < RPT; ++r) {
                    rc0[r] = m[r].x - (v0 - u[r]);
                    rc1[r] = m[r].y - (v1 - u[r]);
                    hit = lt_or(rc1[r], lim, lt_or(rc0[r], lim, hit));
                }
            } else {
                const bool ok0 = j0 < p.D, ok1 = j0 + 1 < p.D;
#pragma unroll
                for (int r = 0; r < RPT; ++r) {
                    const bool rok = i0 + r < p.S_loc;
                    const double a = m[r].x - (v0 - u[r]);
                    const double b = m[r].y - (v1 - u[r]);
                    rc0[r] = (rok && ok0) ? a : INFINITY;
                    rc1[r] = (rok && ok1) ? b : INFINITY;
                    hit = lt_or(rc1[r], lim, lt_or(rc0[r], lim, hit));
                }
            }
            if (WRITE_RC) {
#pragma unroll
                for (int r = 0; r < RPT; ++r) {
                    if (i0 + r < p.S_loc) {
                        double *o = p.rc_out + (i0 + r) * p.ld_out + j0;
                        if (j0 < p.D) o[0] = rc0[r];
                        if (j0 + 1 < p.D) o[1] = rc1[r];
                    }
                }
            }
            tile_epilogue<RPT>(p, tally, tmin, lim, rc0, rc1, hit, (p.row0 + i0) * id_ld + j0, id_ld);
        };
        uint32_t it = 0;
        for (long long k = 0; k < n_static; ++k, ++it) {
            process(rt, cb, (int)(it % STAGES), it, false);
            rt += d_rt; cb += d_cb;
            if (cb >= p.n_col_blocks) { cb -= p.n_col_blocks; ++rt; }
        }
        if (dynamic) {
            for (;; ++it) {
                const int s = it % STAGES;
                mbar_wait(&full_bar[s], (it / STAGES) & 1);
                const long long t = ticket[s];
                if (t < 0) break;
                const long long trt = t / p.n_col_blocks;
                process(trt, t - trt * p.n_col_blocks, s, it, true);
            }
        }
        // one count and one minimum per CTA reach the header (2 368 same-address atomics per pass otherwise)
        const long long k = warp_min(f64_to_min_key(tmin));
        if (lane_id() == 0) { scratch[warp] = k; scratch[CWARPS + STAGES + warp] = (long long)tally.count; }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        long long m = scratch[0];
        unsigned long long cnt = (unsigned long long)scratch[CWARPS + STAGES];
        for (int w = 1; w < CWARPS; ++w) {
            m = scratch[w] < m ? scratch[w] : m;
            cnt += (unsigned long long)scratch[CWARPS + STAGES + w];
        }
        if (cnt) atomicAdd(&p.sink.hdr->n_violating, cnt);
        atomicMin(&p.sink.hdr->min_rc_key, m);
        if (blockIdx.x == 0) atomicAdd(&p.sink.hdr->n_priced, (unsigned long long)(p.S_loc * p.D));
    }
    __syncthreads();
}

constexpr size_t tma_smem_bytes(int rows, int stages, int cwarps, size_t elem_bytes = sizeof(double)) {
    return (size_t)stages * rows * kBoxCols * elem_bytes + 2 * (size_t)stages * sizeof(uint64_t) +
           2 * (size_t)cwarps * sizeof(long long) + (size_t)stages * sizeof(long long) + 64;   // + tickets, counts
}


// ---------------------------------------------------------------------------------------
// host side: tensor map over a row slab of M
// ---------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *,
                                  const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                  const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

// 2-D map {D columns, S_loc rows}, box {256, rows}, over fp64 M or (T = uint32_t) its lower-bound copy.
// l2_promotion 0..3 = none / 64 / 128 / 256 B.
template <class T>
inline int encode_slab_map(CUtensorMap *map, const T *M, int64_t ld, int64_t S_loc, int64_t D, int rows,
                           int l2_promotion) {
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) return SX_ERR_NO_DEVICE;
    cuuint64_t gdim[2]    = {(cuuint64_t)D, (cuuint64_t)S_loc};
    cuuint64_t gstride[1] = {(cuuint64_t)ld * sizeof(T)};
    cuuint32_t box[2]     = {(cuuint32_t)kBoxCols, (cuuint32_t)rows};
    cuuint32_t estr[2]    = {1, 1};
    const CUtensorMapDataType dt = sizeof(T) == 8 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : CU_TENSOR_MAP_DATA_TYPE_UINT32;
    CUresult r = enc(map, dt, 2, (void *)M, gdim, gstride, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                     (CUtensorMapL2promotion)l2_promotion, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { g_last_cuda_error = (int)r; return SX_ERR_CUDA; }
    return SX_OK;
}

}  // namespace sx

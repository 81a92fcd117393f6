// sx_price.cu -- K4: column-generation pricing pass (sm_100a).
//
// Dense OT:  rc_ij = fl(M_ij - fl(y_dst[j] - y_src[i]))  over a row slab of the fp64 cost
// matrix, replacing `self.mcf.c - self.mcf.A.T @ y` + `np.all(rc >= -tol)`
// (reference net_manager.py:474-497; association fixed by SciPy's csc_matvec, SURVEY.md H4).
// Arc list:  rc_k = c_k - (y[tail_k] - y[head_k]), negated where vbasis_k == -2
// (net_manager.py:293-319).
//
// The pass is HBM-bound (8 B per arc, no reuse, no tensor cores).  The main kernel is a
// persistent, warp-specialised TMA pipeline: one producer lane streams ROWS x 256 fp64
// boxes of M into a STAGES-deep shared-memory ring (cp.async.bulk.tensor + mbarrier
// complete_tx), 8 consumer warps read them back with 128-bit shared loads, keep the sink
// potentials of their two columns in registers and fuse: violator count, min reduced cost,
// and compaction of the violating (rc, arc id) pairs for the top-k selection (sx_topk.cu).
#include "sx_price_tma.cuh"

namespace sx {

// K4a, variant 0: the TMA pipeline as a kernel of its own (sx_price_tma.cuh holds the pass).
template <int ROWS, int STAGES, int CWARPS, int MINB, bool WRITE_RC>
__global__ void __launch_bounds__((CWARPS + 1) * 32, MINB)
price_dense_tma_kernel(const __grid_constant__ CUtensorMap tmap, const DenseParams p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    price_tiles<double, ROWS, STAGES, CWARPS, WRITE_RC>(tmap, p, smem_raw);
}

// ---------------------------------------------------------------------------------------
// K4a, variants 1/2: direct global loads (no shared-memory staging).  VEC = 128-bit loads
// (needs 16 B alignment and even ld); otherwise 64-bit loads, any alignment.  Same tile
// walk and same fused epilogue as the TMA kernel; used as the fallback for odd leading
// dimensions and as the non-TMA comparison point in bench sweeps.
// ---------------------------------------------------------------------------------------
constexpr int kDirectRows    = 8;
constexpr int kDirectThreads = 128;

// streaming loads: read-only path, no L1 allocation, L2 evict-first (each cost is read once)
__device__ __forceinline__ double2 ldg_stream_v2(const double *p, uint64_t pol) {
    double2 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.f64 {%0, %1}, [%2], %3;"
                 : "=d"(r.x), "=d"(r.y)
                 : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ double ldg_stream(const double *p, uint64_t pol) {
    double r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(r) : "l"(p), "l"(pol));
    return r;
}

template <bool VEC, bool WRITE_RC>
__global__ void __launch_bounds__(kDirectThreads)
price_dense_direct_kernel(const double *__restrict__ M, long long ld, const DenseParams p) {
    __shared__ long long scratch[kDirectThreads / 32];
    const int warp = threadIdx.x >> 5;
    const long long total = p.n_row_tiles * p.n_col_blocks;
    const long long G = gridDim.x;
    const uint64_t pol = l2_evict_first_policy();
    double    tmin = INFINITY, lim = INFINITY;
    WarpTally tally;
    long long rt = (long long)blockIdx.x / p.n_col_blocks;
    long long cb = (long long)blockIdx.x - rt * p.n_col_blocks;
    const long long d_rt = G / p.n_col_blocks, d_cb = G - d_rt * p.n_col_blocks;
    constexpr int kGap = VEC ? 1 : 128;
    for (long long t = blockIdx.x; t < total; t += G) {
        const long long i0 = rt * kDirectRows;
        // VEC: columns (2c, 2c+1); scalar: columns (c, c + 128) so each load is coalesced
        const long long j0 = cb * kBoxCols + (VEC ? 2 * threadIdx.x : threadIdx.x);
        const long long j1 = j0 + kGap;
        const bool interior = (cb + 1) * kBoxCols <= p.D && (rt + 1) * kDirectRows <= p.S_loc;
        double rc0[kDirectRows], rc1[kDirectRows];
        bool   hit = false;
        if (interior) {
            const double *src = M + i0 * ld + j0;
            double a[kDirectRows], b[kDirectRows];
#pragma unroll
            for (int r = 0; r < kDirectRows; ++r) {
                if (VEC) { const double2 q = ldg_stream_v2(src + r * ld, pol); a[r] = q.x; b[r] = q.y; }
                else { a[r] = ldg_stream(src + r * ld, pol); b[r] = ldg_stream(src + r * ld + kGap, pol); }
            }
            const double v0 = __ldg(p.y_dst + j0), v1 = __ldg(p.y_dst + j1);
#pragma unroll
            for (int r = 0; r < kDirectRows; ++r) {
                const double ui = __ldg(p.y_src + i0 + r);
                rc0[r] = a[r] - (v0 - ui);
                rc1[r] = b[r] - (v1 - ui);
                hit = lt_or(rc1[r], lim, lt_or(rc0[r], lim, hit));
            }
        } else {
            const bool ok0 = j0 < p.D, ok1 = j1 < p.D;
            const double v0 = ok0 ? __ldg(p.y_dst + j0) : 0.0;
            const double v1 = ok1 ? __ldg(p.y_dst + j1) : 0.0;
#pragma unroll
            for (int r = 0; r < kDirectRows; ++r) {
                const bool rok = i0 + r < p.S_loc;
                const double *src = M + (i0 + r) * ld;
                const double a = (rok && ok0) ? ldg_stream(src + j0, pol) : 0.0;
                const double b = (rok && ok1) ? ldg_stream(src + j1, pol) : 0.0;
                const double ui = rok ? __ldg(p.y_src + i0 + r) : 0.0;
                rc0[r] = (rok && ok0) ? a - (v0 - ui) : INFINITY;
                rc1[r] = (rok && ok1) ? b - (v1 - ui) : INFINITY;
                hit = lt_or(rc1[r], lim, lt_or(rc0[r], lim, hit));
            }
        }
        if (WRITE_RC) {
#pragma unroll
            for (int r = 0; r < kDirectRows; ++r) {
                if (i0 + r < p.S_loc) {
                    if (j0 < p.D) p.rc_out[(i0 + r) * p.ld_out + j0] = rc0[r];
                    if (j1 < p.D) p.rc_out[(i0 + r) * p.ld_out + j1] = rc1[r];
                }
            }
        }
        tile_epilogue<kDirectRows>(p, tally, tmin, lim, rc0, rc1, hit, (p.row0 + i0) * p.id_ld + j0, p.id_ld, kGap);
        rt += d_rt; cb += d_cb;
        if (cb >= p.n_col_blocks) { cb -= p.n_col_blocks; ++rt; }
    }
    warp_flush(p.sink, tally);
    block_min_commit(tmin, p.sink.hdr, scratch, kDirectThreads / 32, warp, (unsigned long long)(p.S_loc * p.D));
}

// ---------------------------------------------------------------------------------------
// K4b: arc-list pricing
// ---------------------------------------------------------------------------------------
constexpr int kArcThreads = 256;
constexpr int kArcPerThread = 4;

__global__ void __launch_bounds__(kArcThreads)
price_arcs_kernel(const double *__restrict__ c, const int32_t *__restrict__ tail,
                  const int32_t *__restrict__ head, const int8_t *__restrict__ vbasis,
                  const double *__restrict__ y, long long E, long long id0, double thr,
                  CandSink sink, double *rc_out) {
    __shared__ long long scratch[kArcThreads / 32];
    const int warp = threadIdx.x >> 5;
    double    tmin = INFINITY, lim = INFINITY;
    WarpTally tally;
    const long long chunk = (long long)kArcThreads * kArcPerThread;
    const long long n_chunks = (E + chunk - 1) / chunk;
    const uint64_t pol = l2_evict_first_policy();
    for (long long ch = blockIdx.x; ch < n_chunks; ch += gridDim.x) {
        double rc[kArcPerThread];
        bool   hit = false;
#pragma unroll
        for (int q = 0; q < kArcPerThread; ++q) {
            const long long k = ch * chunk + (long long)q * kArcThreads + threadIdx.x;
            double v = INFINITY;
            if (k < E) {
                const double ck = ldg_stream(c + k, pol);
                const double yt = __ldg(y + tail[k]);
                const double yh = __ldg(y + head[k]);
                v = ck - (yt - yh);
                if (vbasis != nullptr && vbasis[k] == -2) v = -v;
                if (rc_out != nullptr) rc_out[k] = v;
            }
            rc[q] = v;
            hit = lt_or(v, lim, hit);
        }
        if (!__any_sync(0xffffffffu, hit)) continue;
        bool viol = false;
        if (hit) {
            bool nan = false;
#pragma unroll
            for (int q = 0; q < kArcPerThread; ++q) {
                tmin = rc[q] < tmin ? rc[q] : tmin;
                viol = viol || (rc[q] < thr);
                nan = nan || (rc[q] != rc[q]);
            }
            lim = tmin > thr ? tmin : thr;
            if (nan) atomicOr(&sink.hdr->status, kStatusNanRc);
        }
        if (!__any_sync(0xffffffffu, viol)) continue;
        const long long k0 = id0 + ch * chunk + threadIdx.x;
        emit_violators<kArcPerThread>(
            sink, tally, thr, [&](int q) { return rc[q]; },
            [&](int q) { return k0 + (long long)q * kArcThreads; });
    }
    warp_flush(sink, tally);
    block_min_commit(tmin, sink.hdr, scratch, kArcThreads / 32, warp, (unsigned long long)E);
}

// Vectorised form (16-byte aligned arrays): a thread takes two groups of four CONSECUTIVE arcs, so tail, head and
// status come in as one 128-bit (32-bit) load per group and the costs as two; all sixteen y gathers of the thread
// are issued before the first reduced cost is formed.  The kernel is bound by the latency of those gathers (two
// dependent L2 round trips per arc, 2.9 L2 sectors per arc, DRAM at 15 %): what matters is how many are in
// flight, i.e. loads per thread x resident threads (3 CTAs per SM here; the scalar kernel above holds 103
// registers, 2 CTAs per SM, 8 gathers per thread).
constexpr int kArcVecGroups = 2;
constexpr int kArcVecPerThread = 4 * kArcVecGroups;

__global__ void __launch_bounds__(kArcThreads, 3)
price_arcs_vec_kernel(const double *__restrict__ c, const int32_t *__restrict__ tail,
                      const int32_t *__restrict__ head, const int8_t *__restrict__ vbasis,
                      const double *__restrict__ y, long long E4 /* arcs, multiple of 4 */, long long id0, double thr,
                      CandSink sink, double *rc_out) {
    __shared__ long long scratch[kArcThreads / 32];
    const int warp = threadIdx.x >> 5;
    double    tmin = INFINITY, lim = INFINITY;
    WarpTally tally;
    const long long chunk = (long long)kArcThreads * kArcVecPerThread;
    const long long n_chunks = (E4 + chunk - 1) / chunk;
    const uint64_t pol = l2_evict_first_policy();
    for (long long ch = blockIdx.x; ch < n_chunks; ch += gridDim.x) {
        const long long k0 = ch * chunk + (long long)threadIdx.x * 4;
        int4   t4[kArcVecGroups], h4[kArcVecGroups];
        double cc[kArcVecPerThread];
        int    vb[kArcVecGroups];
        bool   in[kArcVecGroups];
#pragma unroll
        for (int g = 0; g < kArcVecGroups; ++g) {
            const long long k = k0 + (long long)g * kArcThreads * 4;
            in[g] = k < E4;
            t4[g] = h4[g] = make_int4(0, 0, 0, 0);
            vb[g] = 0;
            cc[4 * g] = cc[4 * g + 1] = cc[4 * g + 2] = cc[4 * g + 3] = 0.0;
            if (in[g]) {
                t4[g] = __ldcs(reinterpret_cast<const int4 *>(tail + k));
                h4[g] = __ldcs(reinterpret_cast<const int4 *>(head + k));
                const double2 a = ldg_stream_v2(c + k, pol), b = ldg_stream_v2(c + k + 2, pol);
                cc[4 * g] = a.x; cc[4 * g + 1] = a.y; cc[4 * g + 2] = b.x; cc[4 * g + 3] = b.y;
                if (vbasis != nullptr) vb[g] = __ldcs(reinterpret_cast<const int *>(vbasis + k));
            }
        }
        double yt[kArcVecPerThread], yh[kArcVecPerThread];
#pragma unroll
        for (int g = 0; g < kArcVecGroups; ++g) {
            yt[4 * g] = __ldg(y + t4[g].x); yt[4 * g + 1] = __ldg(y + t4[g].y);
            yt[4 * g + 2] = __ldg(y + t4[g].z); yt[4 * g + 3] = __ldg(y + t4[g].w);
            yh[4 * g] = __ldg(y + h4[g].x); yh[4 * g + 1] = __ldg(y + h4[g].y);
            yh[4 * g + 2] = __ldg(y + h4[g].z); yh[4 * g + 3] = __ldg(y + h4[g].w);
        }
        double rc[kArcVecPerThread];
        bool   hit = false;
#pragma unroll
        for (int e = 0; e < kArcVecPerThread; ++e) {
            const int g = e >> 2;
            double v = cc[e] - (yt[e] - yh[e]);
            if ((signed char)(vb[g] >> (8 * (e & 3))) == -2) v = -v;
            rc[e] = in[g] ? v : INFINITY;
            hit = lt_or(rc[e], lim, hit);
        }
        if (rc_out != nullptr) {
#pragma unroll
            for (int g = 0; g < kArcVecGroups; ++g) {
                const long long k = k0 + (long long)g * kArcThreads * 4;
                if (in[g]) {
                    reinterpret_cast<double2 *>(rc_out + k)[0] = make_double2(rc[4 * g], rc[4 * g + 1]);
                    reinterpret_cast<double2 *>(rc_out + k)[1] = make_double2(rc[4 * g + 2], rc[4 * g + 3]);
                }
            }
        }
        if (!__any_sync(0xffffffffu, hit)) continue;
        bool viol = false;
        if (hit) {
            bool nan = false;
#pragma unroll
            for (int e = 0; e < kArcVecPerThread; ++e) {
                tmin = rc[e] < tmin ? rc[e] : tmin;
                viol = viol || (rc[e] < thr);
                nan = nan || (rc[e] != rc[e]);
            }
            lim = tmin > thr ? tmin : thr;
            if (nan) atomicOr(&sink.hdr->status, kStatusNanRc);
        }
        if (!__any_sync(0xffffffffu, viol)) continue;
        emit_violators<kArcVecPerThread>(
            sink, tally, thr, [&](int e) { return rc[e]; },
            [&](int e) { return id0 + k0 + (long long)(e >> 2) * kArcThreads * 4 + (e & 3); });
    }
    warp_flush(sink, tally);
    block_min_commit(tmin, sink.hdr, scratch, kArcThreads / 32, warp, (unsigned long long)E4);
}

// Start of a pricing pass: header cleared, selection state (histograms, counters) zeroed.
__global__ void __launch_bounds__(256) pass_begin_kernel(sx_price_header *h, SelState *st, unsigned K) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        h->n_violating = 0ull;
        h->min_rc_key  = 0x7fffffffffffffffll;
        h->n_priced    = 0ull;
        h->status      = 0ull;
    }
    if (st == nullptr) return;
    uint4 *w = reinterpret_cast<uint4 *>(st);
    const size_t n16 = sizeof(SelState) / 16;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) {
        w[i] = sel_clear_word(i, K);
    }
}

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
// TMA pipeline shapes selectable at run time (bench sweeps): {rows per box, stages, consumer
// warps, CTAs per SM}.  Shared memory = stages * rows * 2 KB per CTA.
struct TmaShape { int rows, stages, cwarps, ctas_per_sm; };
static const TmaShape kTmaShapes[] = {
    {16, 6, 8, 1}, {16, 6, 16, 1}, {32, 3, 8, 1}, {32, 3, 16, 1}, {16, 7, 16, 1}, {8, 12, 16, 1},
    {16, 3, 8, 2}, {8, 6, 8, 2}, {24, 4, 16, 1}, {20, 5, 16, 1}, {12, 9, 16, 1},
    {12, 4, 8, 2}, {8, 7, 8, 2}, {8, 4, 8, 3},
};
constexpr int kNumTmaShapes = sizeof(kTmaShapes) / sizeof(kTmaShapes[0]);
static int g_tma_l2promo = 3, g_tma_evict_first = 1;    // CU_TENSOR_MAP_L2_PROMOTION_L2_256B, L2 evict-first hint
static int g_tma_shape = 6, g_ctas_per_sm_direct = 16;   // 16 rows x 3 stages, 8 consumer warps, 2 CTAs per SM

template <int ROWS, int STAGES, int CWARPS, int MINB, bool WRITE_RC>
static int launch_tma(const CUtensorMap &map, const DenseParams &p, cudaStream_t st) {
    constexpr size_t smem = tma_smem_bytes(ROWS, STAGES, CWARPS);
    auto kern = price_dense_tma_kernel<ROWS, STAGES, CWARPS, MINB, WRITE_RC>;
    SX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const long long total = p.n_row_tiles * p.n_col_blocks;
    long long grid = (long long)num_sms() * MINB;
    if (grid > total) grid = total;
    if (grid < 1) grid = 1;
    kern<<<(int)grid, (CWARPS + 1) * 32, smem, st>>>(map, p);
    SX_LAUNCH_CHECK();
    return SX_OK;
}

template <bool WRITE_RC>
static int dispatch_tma(int shape, const CUtensorMap &map, const DenseParams &p, cudaStream_t st) {
    switch (shape) {
        case 0: return launch_tma<16, 6, 8, 1, WRITE_RC>(map, p, st);
        case 1: return launch_tma<16, 6, 16, 1, WRITE_RC>(map, p, st);
        case 2: return launch_tma<32, 3, 8, 1, WRITE_RC>(map, p, st);
        case 4: return launch_tma<16, 7, 16, 1, WRITE_RC>(map, p, st);
        case 5: return launch_tma<8, 12, 16, 1, WRITE_RC>(map, p, st);
        case 6: return launch_tma<16, 3, 8, 2, WRITE_RC>(map, p, st);
        case 7: return launch_tma<8, 6, 8, 2, WRITE_RC>(map, p, st);
        case 8: return launch_tma<24, 4, 16, 1, WRITE_RC>(map, p, st);
        case 9: return launch_tma<20, 5, 16, 1, WRITE_RC>(map, p, st);
        case 10: return launch_tma<12, 9, 16, 1, WRITE_RC>(map, p, st);
        case 11: return launch_tma<12, 4, 8, 2, WRITE_RC>(map, p, st);
        case 12: return launch_tma<8, 7, 8, 2, WRITE_RC>(map, p, st);
        case 13: return launch_tma<8, 4, 8, 3, WRITE_RC>(map, p, st);
        default: return launch_tma<32, 3, 16, 1, WRITE_RC>(map, p, st);
    }
}

// High word of x's fp64 bit pattern, rounded toward -inf: as the high half of a double (low half 0) it is
// <= x, or NaN when x is NaN.  Positive values and exact ones (low half 0: +-0, +-inf) truncate; a negative
// value with a nonzero low half steps one unit away from zero (-DBL_MAX and below become -inf); a NaN keeps
// its sign and exponent and gets the quiet bit, so its payload cannot vanish into the dropped half.
__device__ __forceinline__ uint32_t cost_lb_word(double x) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(x);
    const uint32_t hi = (uint32_t)(b >> 32), lo = (uint32_t)b;
    if (x != x) return hi | 0x00080000u;
    return (lo != 0 && (hi >> 31)) ? hi + 1u : hi;
}

// Lower-bound copy of a slab (sx_cost_lb_build): one streaming pass, coalesced rows.
__global__ void __launch_bounds__(256) cost_lb_kernel(const double *__restrict__ M, long long ld, long long S_loc,
                                                      long long D, uint32_t *__restrict__ lb, long long ld_lb) {
    for (long long i = blockIdx.x; i < S_loc; i += gridDim.x) {
        const double *src = M + i * ld;
        uint32_t *dst = lb + i * ld_lb;
        for (long long j = threadIdx.x; j < D; j += blockDim.x) dst[j] = cost_lb_word(__ldcs(src + j));
    }
}

}  // namespace sx

using namespace sx;

extern "C" size_t sx_cost_lb_bytes(int64_t S_loc, int64_t D) {
    if (S_loc <= 0 || D <= 0) return 0;
    return (size_t)S_loc * (size_t)((D + 3) & ~(int64_t)3) * sizeof(uint32_t);
}

extern "C" int sx_cost_lb_build(const double *M, int64_t ld, int64_t S_loc, int64_t D, uint32_t *lb, int64_t ld_lb,
                                void *stream) {
    if (!M || !lb || S_loc < 0 || D <= 0 || ld < D || ld_lb < D) return SX_ERR_INVALID;
    if (((uintptr_t)lb % 16) != 0 || (ld_lb % 4) != 0) return SX_ERR_UNALIGNED;
    if (S_loc == 0) return SX_OK;
    long long grid = (long long)num_sms() * 8;
    if (grid > S_loc) grid = S_loc;
    cost_lb_kernel<<<(int)grid, 256, 0, (cudaStream_t)stream>>>(M, ld, S_loc, D, lb, ld_lb);
    SX_LAUNCH_CHECK();
    return SX_OK;
}

extern "C" int sx_price_set_tma_options(int l2_promotion, int evict_first) {
    if (l2_promotion > 3) return SX_ERR_INVALID;
    if (l2_promotion >= 0) g_tma_l2promo = l2_promotion;
    if (evict_first >= 0) g_tma_evict_first = evict_first ? 1 : 0;
    return SX_OK;
}

extern "C" int sx_price_set_tuning(int tma_shape, int direct_ctas_per_sm) {
    if (tma_shape >= kNumTmaShapes) return SX_ERR_INVALID;
    if (tma_shape >= 0) g_tma_shape = tma_shape;
    if (direct_ctas_per_sm > 0) g_ctas_per_sm_direct = direct_ctas_per_sm;
    return SX_OK;
}

extern "C" size_t sx_select_state_bytes(void) { return sizeof(SelState); }

extern "C" int sx_price_pass_begin(sx_price_header *header, sx_select_state *sel, int64_t K, void *stream) {
    if (!header || K < 0 || K > 0xffffffffll) return SX_ERR_INVALID;
    if (((uintptr_t)sel & 15) != 0) return SX_ERR_UNALIGNED;
    pass_begin_kernel<<<sel ? num_sms() : 1, 256, 0, (cudaStream_t)stream>>>(header, (SelState *)sel, (unsigned)K);
    SX_LAUNCH_CHECK();
    return SX_OK;
}

extern "C" int sx_price_dense_ot(const double *M, int64_t ld, int64_t row0, int64_t S_loc, int64_t D,
                                 const double *y_src, const double *y_dst, double tol,
                                 sx_price_header *header, sx_select_state *sel, double *cand_rc,
                                 int64_t *cand_id, int64_t cand_cap, double *rc_out, int64_t ld_out,
                                 int variant, void *stream) {
    if (!M || !y_src || !y_dst || !header || S_loc < 0 || D <= 0 || ld < D || row0 < 0 || cand_cap < 0)
        return SX_ERR_INVALID;
    if (cand_cap > 0 && (!cand_rc || !cand_id || !sel)) return SX_ERR_INVALID;
    if (rc_out && ld_out < D) return SX_ERR_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    if (S_loc == 0) return SX_OK;
    const bool aligned = ((uintptr_t)M % 16 == 0) && (ld % 2 == 0);
    if (variant < 0) variant = aligned ? 0 : 2;
    if ((variant == 0 || variant == 1) && !aligned) return SX_ERR_UNALIGNED;
    if (variant == 0 && (D >= (1ll << 31) || S_loc >= (1ll << 31))) variant = 1;

    DenseParams p;
    p.y_src = y_src; p.y_dst = y_dst; p.M = M; p.ld = ld; p.S_loc = S_loc; p.D = D; p.row0 = row0; p.id_ld = D;
    p.thr = -tol;
    p.sink.hdr = header; p.sink.sel = (SelState *)sel; p.sink.rc = cand_rc; p.sink.id = (int64_t *)cand_id;
    p.sink.cap = cand_cap;
    p.rc_out = rc_out; p.ld_out = ld_out; p.zero = 0; p.evict_first = (uint32_t)g_tma_evict_first;
    p.dyn_ctr = nullptr;
    p.n_col_blocks = (D + kBoxCols - 1) / kBoxCols;

    int rc = SX_OK;
    if (variant == 0) {
        const int rows = kTmaShapes[g_tma_shape].rows;
        p.n_row_tiles = (S_loc + rows - 1) / rows;
        CUtensorMap map;
        if ((rc = encode_slab_map(&map, M, ld, S_loc, D, rows, g_tma_l2promo)) != SX_OK) return rc;
        rc = rc_out ? dispatch_tma<true>(g_tma_shape, map, p, st) : dispatch_tma<false>(g_tma_shape, map, p, st);
    } else {
        p.n_row_tiles = (S_loc + kDirectRows - 1) / kDirectRows;
        const long long total = p.n_row_tiles * p.n_col_blocks;
        long long grid = (long long)num_sms() * g_ctas_per_sm_direct;
        if (grid > total) grid = total;
        if (variant == 1) {
            if (rc_out) price_dense_direct_kernel<true, true><<<(int)grid, kDirectThreads, 0, st>>>(M, ld, p);
            else        price_dense_direct_kernel<true, false><<<(int)grid, kDirectThreads, 0, st>>>(M, ld, p);
        } else {
            if (rc_out) price_dense_direct_kernel<false, true><<<(int)grid, kDirectThreads, 0, st>>>(M, ld, p);
            else        price_dense_direct_kernel<false, false><<<(int)grid, kDirectThreads, 0, st>>>(M, ld, p);
        }
        SX_LAUNCH_CHECK();
    }
    return rc;
}

extern "C" int sx_price_arcs(const double *c, const int32_t *tail, const int32_t *head,
                             const int8_t *vbasis, const double *y, int64_t E, int64_t id0, double tol,
                             sx_price_header *header, sx_select_state *sel, double *cand_rc,
                             int64_t *cand_id, int64_t cand_cap, double *rc_out, void *stream) {
    if (!c || !tail || !head || !y || !header || E < 0 || cand_cap < 0) return SX_ERR_INVALID;
    if (cand_cap > 0 && (!cand_rc || !cand_id || !sel)) return SX_ERR_INVALID;
    if (E == 0) return SX_OK;
    cudaStream_t st = (cudaStream_t)stream;
    CandSink sink{header, (SelState *)sel, cand_rc, (int64_t *)cand_id, cand_cap};
    // the bulk (a multiple of 4 arcs) through the vectorised kernel when every array is 16-byte aligned ...
    const bool aligned = (((uintptr_t)c | (uintptr_t)tail | (uintptr_t)head | (uintptr_t)rc_out) & 15) == 0 &&
                         (((uintptr_t)vbasis) & 3) == 0;
    long long E4 = aligned ? (E / 4) * 4 : 0;
    if (E4 > 0) {
        const long long chunk = (long long)kArcThreads * kArcVecPerThread;
        long long n_chunks = (E4 + chunk - 1) / chunk;
        long long grid = (long long)num_sms() * 3;
        if (grid > n_chunks) grid = n_chunks;
        price_arcs_vec_kernel<<<(int)grid, kArcThreads, 0, st>>>(c, tail, head, vbasis, y, E4, id0, -tol, sink, rc_out);
        SX_LAUNCH_CHECK();
    }
    // ... and the rest (the last < 4 arcs, or everything when something is unaligned) through the scalar one
    if (E4 < E) {
        const long long rest = E - E4;
        const long long chunk = (long long)kArcThreads * kArcPerThread;
        long long n_chunks = (rest + chunk - 1) / chunk;
        long long grid = (long long)num_sms() * 8;
        if (grid > n_chunks) grid = n_chunks;
        price_arcs_kernel<<<(int)grid, kArcThreads, 0, st>>>(c + E4, tail + E4, head + E4, vbasis ? vbasis + E4 : nullptr, y, rest,
                                                             id0 + E4, -tol, sink, rc_out ? rc_out + E4 : nullptr);
    }
    SX_LAUNCH_CHECK();
    return SX_OK;
}

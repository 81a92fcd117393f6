// sx_prefix.cu -- K1d: the head of the Kruskal order without sorting every arc (sm_100a).
//
// `max_weight_spanning_tree` (reference tree_BI.py:32-59) hands ALL n weights to SciPy, whose
// Kruskal argsorts them all although the tree is complete after the first few N arcs of the order
// (SURVEY.md section 6: last tree arc at sorted rank ~8 N of n = N^2 / 4).  This file produces only
// the first T' >= T arcs of that order -- descending weight, ties by ascending arc id -- which is
// all sx_kruskal needs as long as it finishes inside the prefix (the caller checks and falls back
// to the full argsort otherwise; the tree is identical either way because the prefix of a strict
// total order is unique).
//
//   1. histogram of the top 12 bits (sign + exponent) of every weight's order-preserving image (a
//      streaming pass, 8 B per arc -- or free, when sx_score_ot took it while writing the scores);
//   2. split: one more pass appends every arc above the bin b1 that holds the T-th largest weight to
//      the candidate list and sets the arcs of bin b1 aside; the next 12 bits are histogrammed and
//      filtered on that short list (if bin b1 is too crowded for it, two more passes over all weights);
//   3. the few candidates are sorted by id, then stably by weight (radix argsort, sx_sort.cu), and
//      the tie runs are flipped into the Kruskal order (sx_kruskal_order).
// HBM-bound: 8-16 B per arc (24 B in the crowded-bin case) instead of the ~256 B per arc of the full 8-pass argsort.
#include <utility>
#include <vector>

#include "sx_common.cuh"

namespace sx {

constexpr int kPfThreads = 512;
constexpr int kPfBins    = 4096;
constexpr int kPfSub     = 2;      // sub-histograms per CTA (lanes spread over them): fewer same-address conflicts

struct PrefixCtl {
    unsigned long long n_sel;      // candidates appended by the filter
    unsigned long long above;      // arcs in bins strictly above the threshold bin (level 0, then level 0 + 1)
    unsigned int       b1, b2;     // threshold bin of level 0 / level 1
    unsigned long long n_bnd;      // arcs of bin b1 set aside by the split pass
    unsigned int       pad[8];
    unsigned int       hist[2][kPfBins];
};

// LEVEL 0: digit = bits 63..52 of the image.  LEVEL 1: bits 51..40, only for keys whose level-0 digit is b1.
template <int LEVEL>
__global__ void __launch_bounds__(kPfThreads)
pf_hist_kernel(const double *__restrict__ w, long long n, const PrefixCtl *ctl, unsigned *__restrict__ hist_out) {
    __shared__ unsigned sh[kPfSub][kPfBins];
    for (int i = threadIdx.x; i < kPfSub * kPfBins; i += kPfThreads) (&sh[0][0])[i] = 0;
    __syncthreads();
    const unsigned b1 = LEVEL == 1 ? ctl->b1 : 0u;
    unsigned *mine = sh[threadIdx.x & (kPfSub - 1)];
    // run-length cache: consecutive equal digits cost one shared atomic
    unsigned run_d = 0xffffffffu, run_c = 0;
    auto add = [&](double v) {
        const unsigned long long k = f64_to_sort_key(v);
        unsigned d;
        if (LEVEL == 0) d = (unsigned)(k >> 52);
        else {
            if ((unsigned)(k >> 52) != b1) return;
            d = (unsigned)(k >> 40) & (kPfBins - 1);
        }
        if (d == run_d) { ++run_c; return; }
        if (run_c) atomicAdd(&mine[run_d], run_c);
        run_d = d; run_c = 1;
    };
    const long long n2 = n / 2;
    const double2 *w2 = reinterpret_cast<const double2 *>(w);
    const bool aligned = (reinterpret_cast<uintptr_t>(w) & 15) == 0;
    const long long stride = (long long)gridDim.x * kPfThreads;
    if (aligned) {
        for (long long i = (long long)blockIdx.x * kPfThreads + threadIdx.x; i < n2; i += stride) {
            const double2 v = __ldcs(w2 + i);
            add(v.x); add(v.y);
        }
        if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) add(w[n - 1]);
    } else {
        for (long long i = (long long)blockIdx.x * kPfThreads + threadIdx.x; i < n; i += stride) add(__ldcs(w + i));
    }
    if (run_c) atomicAdd(&mine[run_d], run_c);
    __syncthreads();
    for (int i = threadIdx.x; i < kPfBins; i += kPfThreads) {
        unsigned c = 0;
#pragma unroll
        for (int s = 0; s < kPfSub; ++s) c += sh[s][i];
        if (c) atomicAdd(&hist_out[i], c);
    }
}

// One CTA: the largest bin b with count(bins >= b) >= need, scanning the 4096 bins from the top.
template <int LEVEL>
__global__ void __launch_bounds__(1024) pf_bound_kernel(PrefixCtl *ctl, unsigned long long T) {
    __shared__ unsigned long long s_warp[32];
    __shared__ unsigned s_found;
    const unsigned long long need = LEVEL == 0 ? T : (T > ctl->above ? T - ctl->above : 1ull);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // reversed bin index r = 4095 - bin; thread t owns r = 4 t .. 4 t + 3
    unsigned c[4];
    unsigned long long local = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) { c[q] = ctl->hist[LEVEL][kPfBins - 1 - (4 * threadIdx.x + q)]; local += c[q]; }
    unsigned long long incl = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) s_warp[warp] = incl;
    if (threadIdx.x == 0) s_found = 0xffffffffu;
    __syncthreads();
    unsigned long long before = 0;
    for (int w2 = 0; w2 < warp; ++w2) before += s_warp[w2];
    incl += before;
    unsigned long long cum = incl - local;      // count in bins strictly above this thread's first bin
    // the unique thread where the running count crosses `need`
    if (cum < need && incl >= need) {
        int q = 0;
#pragma unroll
        for (int r = 0; r < 4; ++r)
            if (q == r && cum + c[r] < need) { cum += c[r]; ++q; }
        if (q > 3) q = 3;
        s_found = kPfBins - 1 - (4 * threadIdx.x + q);
        if (LEVEL == 0) { ctl->b1 = s_found; ctl->above = cum; }
        else { ctl->b2 = s_found; ctl->above += cum; }
    }
    __syncthreads();
    if (threadIdx.x == 0 && s_found == 0xffffffffu) {   // fewer than `need` arcs in total: take everything
        if (LEVEL == 0) { ctl->b1 = 0; ctl->above = 0; } else ctl->b2 = 0;
    }
}

// Append every arc whose 24-bit prefix is >= (b1, b2).  Each thread keeps kPfBatch 128-bit loads in
// flight before it looks at any of them.  Selected arcs are staged in shared memory and flushed with
// ONE global reservation per CTA and flush: hundreds of thousands of atomicAdds on the single global
// counter would otherwise serialise in L2 and bound the kernel.
constexpr int kPfBatch = 4;
constexpr int kPfStage = 2048;                 // staged candidates per CTA (32 KB)

__global__ void __launch_bounds__(kPfThreads)
pf_filter_kernel(const double *__restrict__ w, const unsigned long long *__restrict__ ids_in, unsigned long long id_base,
                 long long n, PrefixCtl *ctl, double *__restrict__ cand_w, unsigned long long *__restrict__ cand_id,
                 long long cap) {
    __shared__ double             s_w[kPfStage];
    __shared__ unsigned long long s_id[kPfStage];
    __shared__ unsigned           s_cnt;
    __shared__ unsigned long long s_base;
    const unsigned thr = (ctl->b1 << 12) | ctl->b2;
    const unsigned lt = (1u << lane_id()) - 1u;
    const bool aligned = (reinterpret_cast<uintptr_t>(w) & 15) == 0;
    const long long n2 = aligned ? n / 2 : 0;                    // pairs handled by the vector loop
    const double2 *w2 = reinterpret_cast<const double2 *>(w);
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    auto emit = [&](bool keep, double v, long long id) {
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        if (m == 0) return;
        unsigned base = 0;
        if (lane_id() == 0) base = atomicAdd(&s_cnt, (unsigned)__popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        const unsigned slot = base + __popc(m & lt);
        if (!keep) return;
        const unsigned long long gid = ids_in ? ids_in[id] : id_base + (unsigned long long)id;   // position -> arc id
        if (slot < (unsigned)kPfStage) { s_w[slot] = v; s_id[slot] = gid; }
        else {                                                   // stage full (dense selection): straight to global
            const unsigned long long g = atomicAdd(&ctl->n_sel, 1ull);
            if ((long long)g < cap) { cand_w[g] = v; cand_id[g] = gid; }
        }
    };
    auto flush = [&]() {                                         // whole CTA
        __syncthreads();
        const unsigned c = s_cnt < (unsigned)kPfStage ? s_cnt : (unsigned)kPfStage;
        if (threadIdx.x == 0 && c) s_base = atomicAdd(&ctl->n_sel, (unsigned long long)c);
        __syncthreads();
        for (unsigned q = threadIdx.x; q < c; q += kPfThreads) {
            const long long g = (long long)(s_base + q);
            if (g < cap) { cand_w[g] = s_w[q]; cand_id[g] = s_id[q]; }
        }
        __syncthreads();
        if (threadIdx.x == 0) s_cnt = 0;
        __syncthreads();
    };
    // CTA-uniform trip count (flush holds barriers): the CTA walks blocks of kPfThreads pairs
    const long long n2_blocks = (n2 + kPfThreads - 1) / kPfThreads;
    for (long long blk = blockIdx.x; blk < n2_blocks; blk += (long long)gridDim.x * kPfBatch) {
        double2 v[kPfBatch];
#pragma unroll
        for (int u = 0; u < kPfBatch; ++u) {
            const long long i = (blk + (long long)u * gridDim.x) * kPfThreads + threadIdx.x;
            v[u] = i < n2 ? __ldcs(w2 + i) : make_double2(-INFINITY, -INFINITY);
        }
        bool any = false;
#pragma unroll
        for (int u = 0; u < kPfBatch; ++u)
            any = any || (unsigned)(f64_to_sort_key(v[u].x) >> 40) >= thr || (unsigned)(f64_to_sort_key(v[u].y) >> 40) >= thr;
        if (__any_sync(0xffffffffu, any)) {
#pragma unroll
            for (int u = 0; u < kPfBatch; ++u) {
                const long long i = (blk + (long long)u * gridDim.x) * kPfThreads + threadIdx.x;
                const bool in = i < n2;
                emit(in && (unsigned)(f64_to_sort_key(v[u].x) >> 40) >= thr, v[u].x, 2 * i);
                emit(in && (unsigned)(f64_to_sort_key(v[u].y) >> 40) >= thr, v[u].y, 2 * i + 1);
            }
        }
        // an iteration adds at most 8 * kPfThreads entries; flush while there is still room for a typical one
        if (__syncthreads_or(s_cnt > (unsigned)kPfStage / 2)) flush();    // uniform decision, then barriers
    }
    // tail (odd n) or the whole array when it is not 16-byte aligned
    const long long t0 = 2 * n2, nt = n - t0;
    const long long nt_blocks = (nt + kPfThreads - 1) / kPfThreads;
    for (long long blk = blockIdx.x; blk < nt_blocks; blk += gridDim.x) {
        const long long i = blk * kPfThreads + threadIdx.x;
        double v = 0.0;
        bool keep = false;
        if (i < nt) { v = __ldcs(w + t0 + i); keep = (unsigned)(f64_to_sort_key(v) >> 40) >= thr; }
        emit(keep, v, t0 + i);
        if (__syncthreads_or(s_cnt > (unsigned)kPfStage / 2)) flush();
    }
    flush();
}

// One pass that needs only the level-0 bound: arcs above bin b1 are selected outright, arcs inside bin
// b1 are set aside in a boundary list for the second level, which then works on that (short) list
// instead of streaming all the weights twice more.  Two shared-memory stages, flushed like the filter's.
// Top 32 bits of f64_to_sort_key(v) from the high word of v: exact for every v with the sign bit clear
// (a positive NaN lands in bin 4095 like the all-ones key); negative values, -0.0 and negative NaNs take
// the full conversion.  image32 >> 20 is the level-0 bin.
__device__ __forceinline__ unsigned pf_image32(double v) {
    const int hi = __double2hiint(v);
    if (hi < 0) return (unsigned)(f64_to_sort_key(v) >> 32);
    return (unsigned)hi | 0x80000000u;
}

constexpr int kPfHalf = kPfStage / 2;

__global__ void __launch_bounds__(kPfThreads)
pf_split_kernel(const double *__restrict__ w, unsigned long long id_base, long long n, PrefixCtl *ctl,
                double *__restrict__ cand_w, unsigned long long *__restrict__ cand_id, long long cap,
                double *__restrict__ bnd_w, unsigned long long *__restrict__ bnd_id, long long bnd_cap) {
    __shared__ double             s_w[2][kPfHalf];
    __shared__ unsigned long long s_id[2][kPfHalf];
    __shared__ unsigned           s_cnt[2];
    __shared__ unsigned long long s_base[2];
    const unsigned b1 = ctl->b1;
    const unsigned lt = (1u << lane_id()) - 1u;
    const bool aligned = (reinterpret_cast<uintptr_t>(w) & 15) == 0;
    const long long n2 = aligned ? n / 2 : 0;
    const double2 *w2 = reinterpret_cast<const double2 *>(w);
    if (threadIdx.x < 2) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    // which = 0: selected (bin > b1), 1: boundary (bin == b1)
    auto emit = [&](int which, bool keep, double v, long long id) {
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        if (m == 0) return;
        unsigned base = 0;
        if (lane_id() == 0) base = atomicAdd(&s_cnt[which], (unsigned)__popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        const unsigned slot = base + __popc(m & lt);
        if (!keep) return;
        const unsigned long long gid = id_base + (unsigned long long)id;
        if (slot < (unsigned)kPfHalf) { s_w[which][slot] = v; s_id[which][slot] = gid; }
        else {                                                   // stage full: straight to global
            const unsigned long long g = atomicAdd(which ? &ctl->n_bnd : &ctl->n_sel, 1ull);
            if (which == 0) { if ((long long)g < cap) { cand_w[g] = v; cand_id[g] = gid; } }
            else { if ((long long)g < bnd_cap) { bnd_w[g] = v; bnd_id[g] = gid; } }
        }
    };
    auto flush = [&]() {                                         // whole CTA, both stages
        __syncthreads();
        const unsigned c0 = s_cnt[0] < (unsigned)kPfHalf ? s_cnt[0] : (unsigned)kPfHalf;
        const unsigned c1 = s_cnt[1] < (unsigned)kPfHalf ? s_cnt[1] : (unsigned)kPfHalf;
        if (threadIdx.x == 0 && c0) s_base[0] = atomicAdd(&ctl->n_sel, (unsigned long long)c0);
        if (threadIdx.x == 32 && c1) s_base[1] = atomicAdd(&ctl->n_bnd, (unsigned long long)c1);
        __syncthreads();
        for (unsigned q = threadIdx.x; q < c0; q += kPfThreads) {
            const long long g = (long long)(s_base[0] + q);
            if (g < cap) { cand_w[g] = s_w[0][q]; cand_id[g] = s_id[0][q]; }
        }
        for (unsigned q = threadIdx.x; q < c1; q += kPfThreads) {
            const long long g = (long long)(s_base[1] + q);
            if (g < bnd_cap) { bnd_w[g] = s_w[1][q]; bnd_id[g] = s_id[1][q]; }
        }
        __syncthreads();
        if (threadIdx.x < 2) s_cnt[threadIdx.x] = 0;
        __syncthreads();
    };
    // Hot loop.  A weight's level-0 bin is decided from the high word of the double (pf_image32); every
    // lane packs its hits into bit masks.  Hits are a fraction of a percent of the arcs: a warp with hits
    // in a few lanes lets those lanes reserve their own stage slots; a dense warp runs ONE packed warp
    // scan that reserves the slots of both lists.
    const bool     none_above = b1 >= (unsigned)kPfBins - 1;
    const unsigned sel_lo = none_above ? 0xffffffffu : (b1 + 1) << 20;             // image32 >= sel_lo: bin > b1
    auto put = [&](int which, unsigned slot, double v, long long id) {
        const unsigned long long gid = id_base + (unsigned long long)id;
        if (slot < (unsigned)kPfHalf) { s_w[which][slot] = v; s_id[which][slot] = gid; }
        else {                                                   // stage full: straight to global
            const unsigned long long g = atomicAdd(which ? &ctl->n_bnd : &ctl->n_sel, 1ull);
            if (which == 0) { if ((long long)g < cap) { cand_w[g] = v; cand_id[g] = gid; } }
            else { if ((long long)g < bnd_cap) { bnd_w[g] = v; bnd_id[g] = gid; } }
        }
    };
    const long long n2_blocks = (n2 + kPfThreads - 1) / kPfThreads;
    for (long long blk = blockIdx.x; blk < n2_blocks; blk += (long long)gridDim.x * kPfBatch) {
        double2 v[kPfBatch];
#pragma unroll
        for (int u = 0; u < kPfBatch; ++u) {
            const long long i = (blk + (long long)u * gridDim.x) * kPfThreads + threadIdx.x;
            v[u] = i < n2 ? __ldcs(w2 + i) : make_double2(-INFINITY, -INFINITY);
        }
        unsigned sel = 0, bnd = 0;                               // bit 2u: .x, bit 2u + 1: .y
#pragma unroll
        for (int u = 0; u < kPfBatch; ++u) {
            const long long i = (blk + (long long)u * gridDim.x) * kPfThreads + threadIdx.x;
            if (i < n2) {
                const unsigned ix = pf_image32(v[u].x), iy = pf_image32(v[u].y);
                sel |= (unsigned)(!none_above && ix >= sel_lo) << (2 * u) |
                       (unsigned)(!none_above && iy >= sel_lo) << (2 * u + 1);
                bnd |= (unsigned)((ix >> 20) == b1) << (2 * u) | (unsigned)((iy >> 20) == b1) << (2 * u + 1);
            }
        }
        const unsigned mine = (unsigned)__popc(sel) | ((unsigned)__popc(bnd) << 16);
        const unsigned hit_lanes = __ballot_sync(0xffffffffu, mine != 0);
        if (hit_lanes != 0 && __popc(hit_lanes) <= 8) {
            // sparse (the usual case: well under one hit per warp and load batch): only the lanes that hold
            // a hit run, each reserving its stage slots itself
            if (mine) {
#pragma unroll
                for (int u = 0; u < kPfBatch; ++u) {
                    if (((sel | bnd) >> (2 * u)) & 3u) {
                        const long long i = (blk + (long long)u * gridDim.x) * kPfThreads + threadIdx.x;
                        if ((sel >> (2 * u)) & 1u) put(0, atomicAdd(&s_cnt[0], 1u), v[u].x, 2 * i);
                        else if ((bnd >> (2 * u)) & 1u) put(1, atomicAdd(&s_cnt[1], 1u), v[u].x, 2 * i);
                        if ((sel >> (2 * u + 1)) & 1u) put(0, atomicAdd(&s_cnt[0], 1u), v[u].y, 2 * i + 1);
                        else if ((bnd >> (2 * u + 1)) & 1u) put(1, atomicAdd(&s_cnt[1], 1u), v[u].y, 2 * i + 1);
                    }
                }
            }
        } else if (hit_lanes != 0) {
            unsigned incl = mine;                                // packed inclusive scan: <= 256 hits per list and warp
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane_id() >= (unsigned)o) incl += t;
            }
            const unsigned tot = __shfl_sync(0xffffffffu, incl, 31);
            unsigned base0 = 0, base1 = 0;
            if (lane_id() == 31) {
                if (tot & 0xffffu) base0 = atomicAdd(&s_cnt[0], tot & 0xffffu);
                if (tot >> 16) base1 = atomicAdd(&s_cnt[1], tot >> 16);
            }
            base0 = __shfl_sync(0xffffffffu, base0, 31);
            base1 = __shfl_sync(0xffffffffu, base1, 31);
            if (mine) {
                unsigned slot0 = base0 + ((incl - mine) & 0xffffu), slot1 = base1 + ((incl - mine) >> 16);
#pragma unroll
                for (int u = 0; u < kPfBatch; ++u) {
                    const long long i = (blk + (long long)u * gridDim.x) * kPfThreads + threadIdx.x;
                    if ((sel >> (2 * u)) & 1u) put(0, slot0++, v[u].x, 2 * i);
                    if ((bnd >> (2 * u)) & 1u) put(1, slot1++, v[u].x, 2 * i);
                    if ((sel >> (2 * u + 1)) & 1u) put(0, slot0++, v[u].y, 2 * i + 1);
                    if ((bnd >> (2 * u + 1)) & 1u) put(1, slot1++, v[u].y, 2 * i + 1);
                }
            }
        }
        if (__syncthreads_or(s_cnt[0] > (unsigned)kPfHalf / 2 || s_cnt[1] > (unsigned)kPfHalf / 2)) flush();
    }
    const long long t0 = 2 * n2, nt = n - t0;
    const long long nt_blocks = (nt + kPfThreads - 1) / kPfThreads;
    for (long long blk = blockIdx.x; blk < nt_blocks; blk += gridDim.x) {
        const long long i = blk * kPfThreads + threadIdx.x;
        double v = 0.0;
        unsigned b = 0;
        const bool in = i < nt;
        if (in) { v = __ldcs(w + t0 + i); b = (unsigned)(f64_to_sort_key(v) >> 52); }
        emit(0, in && b > b1, v, t0 + i);
        emit(1, in && b == b1, v, t0 + i);
        if (__syncthreads_or(s_cnt[0] > (unsigned)kPfHalf / 2 || s_cnt[1] > (unsigned)kPfHalf / 2)) flush();
    }
    flush();
}

__global__ void pf_gather_kernel(const double *__restrict__ w, const unsigned long long *__restrict__ id,
                                 const uint32_t *__restrict__ perm, long long n, double *w_out, uint32_t *id_out) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const uint32_t s = perm[i];
        w_out[i] = w[s];
        id_out[i] = (uint32_t)id[s];
    }
}
__global__ void pf_gather_ids_kernel(const uint32_t *__restrict__ id, const uint32_t *__restrict__ perm, long long n,
                                     uint32_t *id_out) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        id_out[i] = id[perm[i]];
}

constexpr size_t kPfBndFactor = 4;     // boundary list capacity = 4 x T_cap arcs of the threshold bin

static int pf_grid(long long n, int per_thread) {
    long long g = (n + (long long)kPfThreads * per_thread - 1) / ((long long)kPfThreads * per_thread);
    if (g > num_sms() * 4) g = num_sms() * 4;
    if (g < 1) g = 1;
    return (int)g;
}

// Grids of the split and filter passes over cnt weights on the current device: one wave of resident CTAs at most.
static int pf_pass_grid(const void *kernel, long long cnt) {
    int occ = 1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, kPfThreads, 0) != cudaSuccess || occ < 1) occ = 1;
    const long long ctas = (long long)num_sms() * occ;
    long long need = (cnt / 2 + (long long)kPfThreads * kPfBatch - 1) / ((long long)kPfThreads * kPfBatch);
    if (need < 1) need = 1;
    return (int)(need < ctas ? need : ctas);
}

// The sort-and-order tail shared by sx_kruskal_prefix and sx_order_head_sharded_h: the m <= cap candidates
// (weight, arc id) are sorted by id, then stably by weight (ascending weight, ties by ascending id), and the
// ascending order is turned into the Kruskal order (uint32 ids, descending weight, ties by ascending id) or
// reversed into the queue order (int64 ids, descending weight, ties by descending id).
static size_t pf_tail_bytes(int64_t cap) {
    const size_t c = (size_t)cap;
    return 2 * carve_bytes(c, 8) + 4 * carve_bytes(c, 4) + align_up(sx_argsort_workspace_bytes(cap), 256) +
           sx_kruskal_order_workspace_bytes(cap);
}

static int pf_order_tail(const double *cand_w, const unsigned long long *cand_id, long long m, int64_t cap, int mode,
                         void *out, void *ws, cudaStream_t st) {
    if (m == 0) return SX_OK;
    Carver cv(ws);
    double *w1 = cv.take<double>(cap);
    double *sorted_w = cv.take<double>(cap);
    uint32_t *id1 = cv.take<uint32_t>(cap);
    uint32_t *perm = cv.take<uint32_t>(cap);
    uint32_t *perm2 = cv.take<uint32_t>(cap);
    uint32_t *order_asc = cv.take<uint32_t>(cap);
    void *sort_ws = cv.base + cv.off;
    const size_t sort_ws_bytes = sx_argsort_workspace_bytes(cap);
    void *ko_ws = (char *)sort_ws + align_up(sort_ws_bytes, 256);
    const size_t ko_ws_bytes = sx_kruskal_order_workspace_bytes(cap);
    // (weight, id) is a strict total order: sort by id, then stably by weight
    int rc = sx_argsort_u64(cand_id, m, 32, perm, nullptr, sort_ws, sort_ws_bytes, st);
    if (rc != SX_OK) return rc;
    const int g2 = pf_grid(m, 1);
    pf_gather_kernel<<<g2, kPfThreads, 0, st>>>(cand_w, cand_id, perm, m, w1, id1);
    SX_LAUNCH_CHECK();
    rc = sx_argsort_f64(w1, m, perm2, sorted_w, sort_ws, sort_ws_bytes, st);
    if (rc != SX_OK) return rc;
    pf_gather_ids_kernel<<<g2, kPfThreads, 0, st>>>(id1, perm2, m, order_asc);
    SX_LAUNCH_CHECK();
    if (mode == SX_ORDER_QUEUE) return sx_queue_from_order(order_asc, m, (int64_t *)out, st);
    return sx_kruskal_order(sorted_w, order_asc, m, (uint32_t *)out, ko_ws, ko_ws_bytes, st);
}

}  // namespace sx

using namespace sx;

extern "C" size_t sx_kruskal_prefix_workspace_bytes(int64_t T_cap) {
    if (T_cap < 0) return 0;
    const size_t c = (size_t)T_cap;
    return carve_bytes(1, sizeof(PrefixCtl)) + carve_bytes(c, 8) + carve_bytes(c, 8) +
           2 * carve_bytes(kPfBndFactor * c, 8) + pf_tail_bytes(T_cap) + 256;
}

// hist[bin] += number of weights whose order-preserving image has top 12 bits == bin (4096 bins).
extern "C" int sx_hist12_f64(const double *weight, int64_t n, uint32_t *hist12, void *stream) {
    if (!weight || !hist12 || n < 0) return SX_ERR_INVALID;
    if (n == 0) return SX_OK;
    pf_hist_kernel<0><<<pf_grid(n, 16), kPfThreads, 0, (cudaStream_t)stream>>>(weight, n, nullptr, hist12);
    SX_LAUNCH_CHECK();
    return SX_OK;
}

extern "C" int sx_kruskal_prefix(const double *weight, int64_t n, int64_t T, int64_t T_cap, const uint32_t *hist12,
                                 uint32_t *korder_out, int64_t *n_prefix_h, void *ws, size_t ws_bytes, void *stream) {
    if (!weight || n <= 0 || T <= 0 || T_cap < T || !korder_out || !n_prefix_h) return SX_ERR_INVALID;
    if (n >= (1ll << 32)) return SX_ERR_TOO_LARGE;
    if (!ws || ws_bytes < sx_kruskal_prefix_workspace_bytes(T_cap)) return SX_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    Carver cv(ws);
    PrefixCtl *ctl = cv.take<PrefixCtl>(1);
    double *cand_w = cv.take<double>(T_cap);
    unsigned long long *cand_id = cv.take<unsigned long long>(T_cap);
    double *bnd_w = cv.take<double>(kPfBndFactor * (size_t)T_cap);
    unsigned long long *bnd_id = cv.take<unsigned long long>(kPfBndFactor * (size_t)T_cap);
    void *tail_ws = cv.base + cv.off;

    SX_CUDA(cudaMemsetAsync(ctl, 0, sizeof(PrefixCtl), st));
    const int grid = pf_grid(n, 16);
    if (hist12) {   // level-0 histogram already taken (sx_score_ot produced it while writing the scores)
        SX_CUDA(cudaMemcpyAsync(ctl->hist[0], hist12, sizeof(unsigned) * kPfBins, cudaMemcpyDeviceToDevice, st));
    } else {
        pf_hist_kernel<0><<<grid, kPfThreads, 0, st>>>(weight, n, ctl, ctl->hist[0]);
        SX_LAUNCH_CHECK();
    }
    pf_bound_kernel<0><<<1, 1024, 0, st>>>(ctl, (unsigned long long)T);
    SX_LAUNCH_CHECK();
    // level 1.  Preferred: ONE more pass over the weights that selects everything above bin b1 and sets
    // the arcs of bin b1 aside; the second histogram and the filter then run on that short list.  If the
    // threshold bin is too crowded for the list, both run over all the weights instead.
    const long long bnd_cap = (long long)(kPfBndFactor * (size_t)T_cap);
    pf_split_kernel<<<pf_pass_grid((const void *)pf_split_kernel, n), kPfThreads, 0, st>>>(
        weight, 0, n, ctl, cand_w, cand_id, T_cap, bnd_w, bnd_id, bnd_cap);
    SX_LAUNCH_CHECK();
    unsigned long long n_bnd = 0;
    SX_CUDA(cudaMemcpyAsync(&n_bnd, &ctl->n_bnd, sizeof(n_bnd), cudaMemcpyDeviceToHost, st));
    SX_CUDA(cudaStreamSynchronize(st));
    const void *filter = (const void *)pf_filter_kernel;
    if (n_bnd <= (unsigned long long)bnd_cap) {
        const long long mb = (long long)n_bnd;
        if (mb > 0) {
            pf_hist_kernel<1><<<pf_grid(mb, 16), kPfThreads, 0, st>>>(bnd_w, mb, ctl, ctl->hist[1]);
            SX_LAUNCH_CHECK();
        }
        pf_bound_kernel<1><<<1, 1024, 0, st>>>(ctl, (unsigned long long)T);
        SX_LAUNCH_CHECK();
        if (mb > 0) {
            pf_filter_kernel<<<pf_pass_grid(filter, mb), kPfThreads, 0, st>>>(bnd_w, bnd_id, 0, mb, ctl, cand_w,
                                                                               cand_id, T_cap);
            SX_LAUNCH_CHECK();
        }
    } else {
        SX_CUDA(cudaMemsetAsync(&ctl->n_sel, 0, sizeof(unsigned long long), st));       // the filter selects from scratch
        pf_hist_kernel<1><<<grid, kPfThreads, 0, st>>>(weight, n, ctl, ctl->hist[1]);
        SX_LAUNCH_CHECK();
        pf_bound_kernel<1><<<1, 1024, 0, st>>>(ctl, (unsigned long long)T);
        SX_LAUNCH_CHECK();
        pf_filter_kernel<<<pf_pass_grid(filter, n), kPfThreads, 0, st>>>(weight, nullptr, 0, n, ctl, cand_w, cand_id,
                                                                          T_cap);
        SX_LAUNCH_CHECK();
    }
    unsigned long long n_sel = 0;
    SX_CUDA(cudaMemcpyAsync(&n_sel, &ctl->n_sel, sizeof(n_sel), cudaMemcpyDeviceToHost, st));
    SX_CUDA(cudaStreamSynchronize(st));
    if (n_sel > (unsigned long long)T_cap) {   // too many ties at the threshold for this capacity
        *n_prefix_h = -1;
        return SX_OK;
    }
    *n_prefix_h = (long long)n_sel;
    return pf_order_tail(cand_w, cand_id, (long long)n_sel, T_cap, SX_ORDER_KRUSKAL, korder_out, tail_ws, st);
}

// ---- row-sharded form (sx_order_head_sharded_h) ------------------------------------------------------------------
namespace {

// One shard of sx_order_head_sharded_h: its weights, control block and candidate / boundary lists, carved from
// one allocation on the shard's device.
struct PfShard {
    int dev = 0;
    cudaStream_t st = nullptr;                 // the stream of this shard's device (shards of one device share it)
    const double *w = nullptr;
    long long n = 0;
    unsigned long long id0 = 0;                // global id of the shard's first weight
    void *mem = nullptr;
    PrefixCtl *ctl = nullptr;
    double *cand_w = nullptr, *bnd_w = nullptr;
    unsigned long long *cand_id = nullptr, *bnd_id = nullptr;
    unsigned long long n_bnd = 0, n_sel = 0;
};

struct PfSharded {
    std::vector<PfShard> r;
    std::vector<std::pair<int, cudaStream_t>> streams;   // one per distinct device
    void *mem0 = nullptr;                                // gathered candidates + tail workspace, on r[0].dev
    int prev = 0;
    ~PfSharded() {
        for (auto &ds : streams) {
            cudaSetDevice(ds.first);
            cudaStreamSynchronize(ds.second);
            cudaStreamDestroy(ds.second);
        }
        for (PfShard &k : r) {
            if (!k.mem) continue;
            cudaSetDevice(k.dev);
            cudaFree(k.mem);
        }
        if (mem0) { cudaSetDevice(r[0].dev); cudaFree(mem0); }
        cudaSetDevice(prev);
    }
    int sync() {
        for (auto &ds : streams) {
            SX_CUDA(cudaSetDevice(ds.first));
            SX_CUDA(cudaStreamSynchronize(ds.second));
        }
        return SX_OK;
    }
    // Sums the shards' level-LEVEL histograms on the host (S * D < 2^32: uint32 bins hold every count), writes the
    // sum back into every shard's control block and finds the threshold bin there: every shard sees the same bound.
    template <int LEVEL> int merge_hist(int64_t T, std::vector<unsigned> &h) {
        const size_t G = r.size(), bytes = sizeof(unsigned) * kPfBins;
        h.assign((G + 1) * kPfBins, 0u);
        for (size_t g = 0; g < G; ++g) {
            SX_CUDA(cudaSetDevice(r[g].dev));
            SX_CUDA(cudaMemcpyAsync(&h[(g + 1) * kPfBins], r[g].ctl->hist[LEVEL], bytes, cudaMemcpyDeviceToHost, r[g].st));
        }
        int rc = sync();
        if (rc != SX_OK) return rc;
        for (size_t g = 0; g < G; ++g)
            for (int b = 0; b < kPfBins; ++b) h[b] += h[(g + 1) * kPfBins + b];
        for (PfShard &k : r) {
            SX_CUDA(cudaSetDevice(k.dev));
            SX_CUDA(cudaMemcpyAsync(k.ctl->hist[LEVEL], h.data(), bytes, cudaMemcpyHostToDevice, k.st));
            pf_bound_kernel<LEVEL><<<1, 1024, 0, k.st>>>(k.ctl, (unsigned long long)T);
            SX_LAUNCH_CHECK();
        }
        return SX_OK;
    }
};

}  // namespace

extern "C" int sx_order_head_sharded_h(int ndev, const int *devs, const double *const *weights,
                                       const int64_t *row_bounds, int64_t S, int64_t D, int64_t T, int64_t T_cap,
                                       const uint32_t *const *hist12, int mode, void *out, int64_t *n_out_h) {
    if (ndev < 1 || ndev > 64 || !devs || !weights || S < 1 || D < 1 || ndev > S || T < 1 || T_cap < T || !out ||
        !n_out_h || (mode != SX_ORDER_KRUSKAL && mode != SX_ORDER_QUEUE))
        return SX_ERR_INVALID;
    if (row_bounds) {
        if (row_bounds[0] != 0 || row_bounds[ndev] != S) return SX_ERR_INVALID;
        for (int g = 0; g < ndev; ++g) if (row_bounds[g + 1] <= row_bounds[g]) return SX_ERR_INVALID;
    }
    for (int g = 0; g < ndev; ++g) if (!weights[g]) return SX_ERR_INVALID;
    if (S >= (1ll << 32) || D >= (1ll << 32) || (unsigned long long)S * (unsigned long long)D >= (1ull << 32))
        return SX_ERR_TOO_LARGE;
    const long long n = S * D;
    if (T > n) T = n;
    const int G = ndev;
    const long long bnd_cap = (long long)(kPfBndFactor * (size_t)T_cap);
    PfSharded sh;
    SX_CUDA(cudaGetDevice(&sh.prev));
    sh.r.resize(G);
    for (int g = 0; g < G; ++g) {
        PfShard &k = sh.r[g];
        k.dev = devs[g];
        k.w = weights[g];
        const long long row0 = row_bounds ? row_bounds[g] : S * g / G;
        k.n = ((row_bounds ? row_bounds[g + 1] : S * (g + 1) / G) - row0) * D;
        k.id0 = (unsigned long long)(row0 * D);
        if (cudaSetDevice(k.dev) != cudaSuccess) return SX_ERR_NO_DEVICE;
        for (auto &ds : sh.streams) if (ds.first == k.dev) k.st = ds.second;
        if (!k.st) {
            SX_CUDA(cudaStreamCreateWithFlags(&k.st, cudaStreamNonBlocking));
            sh.streams.emplace_back(k.dev, k.st);
        }
        SX_CUDA(cudaMalloc(&k.mem, carve_bytes(1, sizeof(PrefixCtl)) + 2 * carve_bytes((size_t)T_cap, 8) +
                                       2 * carve_bytes((size_t)bnd_cap, 8)));
        Carver cv(k.mem);
        k.ctl = cv.take<PrefixCtl>(1);
        k.cand_w = cv.take<double>(T_cap);
        k.cand_id = cv.take<unsigned long long>(T_cap);
        k.bnd_w = cv.take<double>(bnd_cap);
        k.bnd_id = cv.take<unsigned long long>(bnd_cap);
        // level 0: the shard's histogram (or the one sx_score_ot took while writing the scores)
        SX_CUDA(cudaMemsetAsync(k.ctl, 0, sizeof(PrefixCtl), k.st));
        if (hist12 && hist12[g]) {
            SX_CUDA(cudaMemcpyAsync(k.ctl->hist[0], hist12[g], sizeof(unsigned) * kPfBins, cudaMemcpyDeviceToDevice,
                                    k.st));
        } else {
            pf_hist_kernel<0><<<pf_grid(k.n, 16), kPfThreads, 0, k.st>>>(k.w, k.n, k.ctl, k.ctl->hist[0]);
            SX_LAUNCH_CHECK();
        }
    }
    std::vector<unsigned> h;
    int rc = sh.merge_hist<0>(T, h);
    if (rc != SX_OK) return rc;
    // split pass on every shard, then each shard's level-1 histogram: on its boundary list, or on all its weights
    // when the list overflowed (each shard decides for itself; the filter then selects that shard from scratch)
    for (PfShard &k : sh.r) {
        SX_CUDA(cudaSetDevice(k.dev));
        pf_split_kernel<<<pf_pass_grid((const void *)pf_split_kernel, k.n), kPfThreads, 0, k.st>>>(
            k.w, k.id0, k.n, k.ctl, k.cand_w, k.cand_id, T_cap, k.bnd_w, k.bnd_id, bnd_cap);
        SX_LAUNCH_CHECK();
    }
    for (PfShard &k : sh.r) {
        SX_CUDA(cudaSetDevice(k.dev));
        SX_CUDA(cudaMemcpyAsync(&k.n_bnd, &k.ctl->n_bnd, sizeof(k.n_bnd), cudaMemcpyDeviceToHost, k.st));
    }
    if ((rc = sh.sync()) != SX_OK) return rc;
    for (PfShard &k : sh.r) {
        SX_CUDA(cudaSetDevice(k.dev));
        if (k.n_bnd <= (unsigned long long)bnd_cap) {
            if (k.n_bnd > 0)
                pf_hist_kernel<1><<<pf_grid((long long)k.n_bnd, 16), kPfThreads, 0, k.st>>>(k.bnd_w, (long long)k.n_bnd,
                                                                                          k.ctl, k.ctl->hist[1]);
        } else {
            SX_CUDA(cudaMemsetAsync(&k.ctl->n_sel, 0, sizeof(unsigned long long), k.st));
            pf_hist_kernel<1><<<pf_grid(k.n, 16), kPfThreads, 0, k.st>>>(k.w, k.n, k.ctl, k.ctl->hist[1]);
        }
        SX_LAUNCH_CHECK();
    }
    if ((rc = sh.merge_hist<1>(T, h)) != SX_OK) return rc;
    const void *filter = (const void *)pf_filter_kernel;
    for (PfShard &k : sh.r) {
        SX_CUDA(cudaSetDevice(k.dev));
        if (k.n_bnd <= (unsigned long long)bnd_cap) {
            const long long mb = (long long)k.n_bnd;
            if (mb > 0)
                pf_filter_kernel<<<pf_pass_grid(filter, mb), kPfThreads, 0, k.st>>>(k.bnd_w, k.bnd_id, 0, mb, k.ctl,
                                                                                     k.cand_w, k.cand_id, T_cap);
        } else {
            pf_filter_kernel<<<pf_pass_grid(filter, k.n), kPfThreads, 0, k.st>>>(k.w, nullptr, k.id0, k.n, k.ctl,
                                                                                  k.cand_w, k.cand_id, T_cap);
        }
        SX_LAUNCH_CHECK();
        SX_CUDA(cudaMemcpyAsync(&k.n_sel, &k.ctl->n_sel, sizeof(k.n_sel), cudaMemcpyDeviceToHost, k.st));
    }
    if ((rc = sh.sync()) != SX_OK) return rc;
    unsigned long long m = 0;
    for (PfShard &k : sh.r) m += k.n_sel;          // a shard over T_cap puts the sum over T_cap too
    if (m > (unsigned long long)T_cap) {           // too many ties at the threshold for this capacity
        *n_out_h = -1;
        return SX_OK;
    }
    // the candidates of every shard go to devs[0] (at most T_cap of them), where they are sorted and ordered
    PfShard &k0 = sh.r[0];
    SX_CUDA(cudaSetDevice(k0.dev));
    SX_CUDA(cudaMalloc(&sh.mem0, 2 * carve_bytes((size_t)T_cap, 8) + pf_tail_bytes(T_cap) + 256));
    Carver cv(sh.mem0);
    double *all_w = cv.take<double>(T_cap);
    unsigned long long *all_id = cv.take<unsigned long long>(T_cap);
    void *tail_ws = cv.base + cv.off;
    unsigned long long off = 0;
    for (PfShard &k : sh.r) {
        if (k.n_sel == 0) continue;
        if (k.dev == k0.dev) {
            SX_CUDA(cudaMemcpyAsync(all_w + off, k.cand_w, k.n_sel * 8, cudaMemcpyDeviceToDevice, k0.st));
            SX_CUDA(cudaMemcpyAsync(all_id + off, k.cand_id, k.n_sel * 8, cudaMemcpyDeviceToDevice, k0.st));
        } else {
            SX_CUDA(cudaMemcpyPeerAsync(all_w + off, k0.dev, k.cand_w, k.dev, k.n_sel * 8, k0.st));
            SX_CUDA(cudaMemcpyPeerAsync(all_id + off, k0.dev, k.cand_id, k.dev, k.n_sel * 8, k0.st));
        }
        off += k.n_sel;
    }
    rc = pf_order_tail(all_w, all_id, (long long)m, T_cap, mode, out, tail_ws, k0.st);
    if (rc != SX_OK) return rc;
    SX_CUDA(cudaStreamSynchronize(k0.st));
    *n_out_h = (long long)m;
    return SX_OK;
}

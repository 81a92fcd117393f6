// sx_sinkhorn.cu -- interior-point warm start for optimal transport: entropic Sinkhorn iterations in
// the log domain on the dense cost matrix (sm_100a).
//
// The reference's experiment driver produces the first-order point it then crosses over with POT:
// `sinkhorn_x = sinkhorn(ot.s, ot.d, ot.M, reg=10, numItermax=1000)` (scripts/run_network_crossover.py:96),
// i.e. Sinkhorn-Knopp  u = a / (K v),  v = b / (K^T u),  K = exp(-M / reg),  X = diag(u) K diag(v),
// stopping when the column-marginal error drops below stopThr (checked every 10 iterations).  POT is a
// third-party package that is not in the reference tree (and not installable offline); this file
// restates the same iteration (same order: v first, from u = 1 / S) with potentials f = reg log u,
// g = reg log v, which is the identical map in exact arithmetic and does not overflow for small reg:
//     g_j = reg log b_j - reg LSE_i((f_i - M_ij) / reg)
//     f_i = reg log a_i - reg LSE_j((g_j - M_ij) / reg)
//     X_ij = exp((f_i + g_j - M_ij) / reg)
// Streaming passes over M: one per half-iteration (8 B per arc) with an online (running max, scaled
// sum) log-sum-exp taken in groups of 8 arcs per thread, plus one read + one write for X at the end.
// The column-marginal error of POT's test is free: with the new f and the old g the column sums of X
// are b_j exp((g_old_j - g_new_j) / reg), so the error of iteration k is known during the column pass
// of iteration k + 1 (the loop then stops with that pass's g, one half-step further than POT).
// sx_sinkhorn_ot_sharded_h runs the same kernels on row slabs spread over several GPUs (the shards sx_ot_pricer
// prices): the row half-step reads only a slab's own rows; the column half-step exchanges one log-sum-exp pair
// per column and rank over NVLink (push / fold kernels below) and merges the pairs in rank order on every rank.
#include <math.h>
#include <string.h>

#include <vector>

#include "sx_common.cuh"
#include "sx_expm.cuh"
#include "sx_ll.cuh"

namespace sx {

// The two streaming passes were instruction-issue and fp64-pipe bound, not HBM bound (round-2 capture of
// the first version, profiles/r02_sinkhorn_raw.csv: 84 % issue slots, 91 warp instructions per arc, fp64
// pipe 52 %, DRAM 33 %): one libm exp per arc plus a second one whenever ANY lane of the warp met a new
// running maximum.  They now take the arcs in groups of kSkGroup per thread -- loads first (kSkGroup
// independent 8-byte loads in flight), one shared maximum per group, one rescale of the running sum per
// group, and the sign-aware 11-operation exp of sx_expm.cuh -- ~17 fp64 operations per arc and no
// divergent branch.
constexpr int kSkGroup = 8;

__constant__ double c_exp_tab[kExpTabSize] = {SX_EXP_TAB_VALUES};

__device__ __forceinline__ void load_exp_tab(double *s_tab) {      // all threads of the CTA call this
    if (threadIdx.x < kExpTabSize) s_tab[threadIdx.x] = c_exp_tab[threadIdx.x];
    __syncthreads();
}

struct Lse {          // log-sum-exp accumulator: sum of exp(t_k) = s * exp(m)
    double m, s;
};
// Accumulation works on the unscaled w_k = potential - cost (t_k = w_k / reg): `wm` is the running
// maximum of w, acc.m = wm / reg rounded once, and every exponent is fma(w_k, 1 / reg, -acc.m).
__device__ __forceinline__ void lse_add_group(Lse &a, double &wm, const double (&w)[kSkGroup], double inv,
                                              const double *tab) {
    double gm = w[0];
#pragma unroll
    for (int k = 1; k < kSkGroup; ++k) gm = w[k] > gm ? w[k] : gm;
    gm = gm > wm ? gm : wm;
    if (gm == -INFINITY) return;                      // only masked slots so far
    const double q = gm * inv;
    double s = a.s * exp_nonpos(a.m - q, tab);        // a.m = -inf: exp gives 0 (and a.s is 0)
    const double nq = -q;
#pragma unroll
    for (int k = 0; k < kSkGroup; ++k) s += exp_nonpos(fma(w[k], inv, nq), tab);   // masked slots (-inf) add 0
    wm = gm;
    a.m = q;
    a.s = s;
}
__device__ __forceinline__ void lse_merge(Lse &a, const Lse &b) {
    if (b.m <= a.m) a.s += b.s * exp(b.m - a.m);
    else { a.s = a.s * exp(a.m - b.m) + b.s; a.m = b.m; }
}
// merge of partial accumulators; an empty one (s = 0: masked slots only, or every term underflowed) is skipped
__device__ __forceinline__ void lse_fold(Lse &acc, const Lse &other) {
    if (other.s > 0.0) { if (acc.s > 0.0) lse_merge(acc, other); else acc = other; }
}

// f update: one warp per row, lanes stride the columns (coalesced), kSkGroup * 32 columns per step.
__global__ void __launch_bounds__(256)
sk_row_kernel(const double *__restrict__ M, long long ld, long long S, long long D, const double *__restrict__ g,
              const double *__restrict__ log_a, double reg, double *__restrict__ f) {
    __shared__ double s_tab[kExpTabSize];
    load_exp_tab(s_tab);
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
    const int lane = lane_id();
    const double inv = 1.0 / reg;
    constexpr long long kStep = (long long)kSkGroup * 32;
    for (long long i = warp; i < S; i += n_warps) {
        const double *row = M + i * ld;
        Lse acc{-INFINITY, 0.0};
        double wm = -INFINITY;
        long long j0 = 0;
        double nx[kSkGroup];                          // the next group's costs, in flight during this group's math
        if (kStep <= D) {
#pragma unroll
            for (int k = 0; k < kSkGroup; ++k) nx[k] = __ldcs(row + lane + 32 * k);
        }
        for (; j0 + kStep <= D; j0 += kStep) {
            double w[kSkGroup];
#pragma unroll
            for (int k = 0; k < kSkGroup; ++k) w[k] = g[j0 + lane + 32 * k] - nx[k];
            if (j0 + 2 * kStep <= D) {
#pragma unroll
                for (int k = 0; k < kSkGroup; ++k) nx[k] = __ldcs(row + j0 + kStep + lane + 32 * k);
            }
            lse_add_group(acc, wm, w, inv, s_tab);
        }
        if (j0 < D) {
            double w[kSkGroup];
#pragma unroll
            for (int k = 0; k < kSkGroup; ++k) {
                const long long j = j0 + lane + 32 * k;
                w[k] = j < D ? g[j] - __ldcs(row + j) : -INFINITY;
            }
            lse_add_group(acc, wm, w, inv, s_tab);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            Lse other{__shfl_xor_sync(0xffffffffu, acc.m, o), __shfl_xor_sync(0xffffffffu, acc.s, o)};
            if (other.s > 0.0) { if (acc.s > 0.0) lse_merge(acc, other); else acc = other; }
        }
        if (lane == 0) f[i] = reg * (log_a[i] - (acc.m + log(acc.s)));
    }
}

// g update, stage 1: a CTA covers 256 columns x `rows_per_chunk` rows; partial LSE per (chunk, column).
__global__ void __launch_bounds__(256)
sk_col_partial_kernel(const double *__restrict__ M, long long ld, long long S, long long D,
                      const double *__restrict__ f, double reg, long long rows_per_chunk,
                      double *__restrict__ pm, double *__restrict__ ps) {
    __shared__ double s_tab[kExpTabSize];
    load_exp_tab(s_tab);
    const long long j = (long long)blockIdx.x * 256 + threadIdx.x;
    const long long chunk = blockIdx.y;
    const long long i0 = chunk * rows_per_chunk, i1 = i0 + rows_per_chunk < S ? i0 + rows_per_chunk : S;
    if (j >= D) return;
    const double inv = 1.0 / reg;
    const double *col = M + j;
    Lse acc{-INFINITY, 0.0};
    double wm = -INFINITY;
    long long i = i0;
    double nx[kSkGroup];                              // the next group's costs, in flight during this group's math
    if (i + kSkGroup <= i1) {
#pragma unroll
        for (int k = 0; k < kSkGroup; ++k) nx[k] = __ldcs(col + (i + k) * ld);
    }
    for (; i + kSkGroup <= i1; i += kSkGroup) {
        double w[kSkGroup];
#pragma unroll
        for (int k = 0; k < kSkGroup; ++k) w[k] = f[i + k] - nx[k];
        if (i + 2 * kSkGroup <= i1) {
#pragma unroll
            for (int k = 0; k < kSkGroup; ++k) nx[k] = __ldcs(col + (i + kSkGroup + k) * ld);
        }
        lse_add_group(acc, wm, w, inv, s_tab);
    }
    if (i < i1) {
        double w[kSkGroup];
#pragma unroll
        for (int k = 0; k < kSkGroup; ++k) w[k] = i + k < i1 ? f[i + k] - __ldcs(col + (i + k) * ld) : -INFINITY;
        lse_add_group(acc, wm, w, inv, s_tab);
    }
    pm[chunk * D + j] = acc.m;
    ps[chunk * D + j] = acc.s;
}

// g update, stage 2, first job: the chunk partials of column j merged in chunk order (empty partials, s = 0, skipped).
__device__ __forceinline__ Lse sk_merge_chunks(long long D, long long n_chunks, const double *__restrict__ pm,
                                               const double *__restrict__ ps, long long j) {
    Lse acc{-INFINITY, 0.0};
    for (long long c = 0; c < n_chunks; ++c) lse_fold(acc, Lse{pm[c * D + j], ps[c * D + j]});
    return acc;
}

// g update, stage 2, second job: g_j = reg (log b_j - LSE_j); returns the term (b_j (exp((g_old - g_new)/reg) - 1))^2
// of POT's error.
__device__ __forceinline__ double sk_col_finish(const Lse &acc, double log_b, double b, double reg, double &g) {
    const double g_new = reg * (log_b - (acc.m + log(acc.s)));
    const double e = b * (exp((g - g_new) / reg) - 1.0);
    g = g_new;
    return e * e;
}

// Sum of the error terms of a 256-thread CTA, in a fixed order; valid in thread 0.  Every thread of the CTA calls it.
__device__ __forceinline__ double sk_err_block_sum(double e2) {
    __shared__ double s_err[8];
    e2 = warp_sum(e2);
    if (lane_id() == 0) s_err[threadIdx.x >> 5] = e2;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x == 0)
        for (int w = 0; w < 8; ++w) t += s_err[w];
    return t;
}

// g update, stage 2: merge the chunks of a column; accumulate POT's error sum_j (b_j (exp((g_old - g_new)/reg) - 1))^2.
__global__ void __launch_bounds__(256)
sk_col_merge_kernel(long long D, long long n_chunks, const double *__restrict__ pm, const double *__restrict__ ps,
                    const double *__restrict__ log_b, const double *__restrict__ b, double reg,
                    double *__restrict__ g, double *err2) {
    const long long j = (long long)blockIdx.x * 256 + threadIdx.x;
    double e2 = 0.0;
    if (j < D) e2 = sk_col_finish(sk_merge_chunks(D, n_chunks, pm, ps, j), log_b[j], b[j], reg, g[j]);
    const double t = sk_err_block_sum(e2);
    if (threadIdx.x == 0 && err2 != nullptr && t != 0.0) atomicAdd(err2, t);
}

// ---- row-sharded form (sx_sinkhorn_ot_sharded_h) ------------------------------------------------------------
// Rank r holds rows [row0_r, row0_r + S_loc_r) of M and runs the kernels above on them; f is local to the rank,
// g is computed by every rank.  The column half-step needs one (m, s) pair per column from every rank: the push
// kernel merges the rank's chunk partials and stores the pair into every rank's exchange buffer as two LL slots
// (sx_ll.cuh; block_len = 2 D slots per rank, flag = iteration + 1, half = flag & 1); the fold kernel polls the
// G pairs of its column in the local buffer and merges them in rank order, so every rank computes the same g.
// Double buffering suffices: a rank pushes iteration e + 1 only after its own fold of e, which needed every
// peer's push of e, which that peer enqueued after its fold of e - 1 -- the last reader of the same half.
__global__ void __launch_bounds__(256)
sk_col_push_kernel(long long D, long long n_chunks, const double *__restrict__ pm, const double *__restrict__ ps,
                   char *const *peer_bufs, int rank, int G, unsigned flag) {
    const long long j = (long long)blockIdx.x * 256 + threadIdx.x;
    if (j >= D) return;
    const Lse acc = sk_merge_chunks(D, n_chunks, pm, ps, j);
    for (int p = 0; p < G; ++p) {
        uint4 *dst = ll_slot(peer_bufs[p], G, 2 * D, flag, rank, 2 * j);
        ll_store_slot(dst, flag, (unsigned long long)__double_as_longlong(acc.m));
        ll_store_slot(dst + 1, flag, (unsigned long long)__double_as_longlong(acc.s));
    }
}

// err_part (may be null): CTA c writes the sum of its columns' error terms to err_part[c], and the host adds them
// in CTA order -- unlike an atomic sum, the error (and so the iteration a run stops at) does not depend on the
// order in which CTAs finish, which differs between ranks sharing a GPU and ranks waiting on NVLink peers.
// status: SX_ERR_PEER_TIMEOUT when some pair did not arrive within timeout_ns; once it is set, later folds return
// at once (g is then stale and the host reports the error).
__global__ void __launch_bounds__(256)
sk_col_fold_kernel(long long D, char *ll_local, int G, unsigned flag, const double *__restrict__ log_b,
                   const double *__restrict__ b, double reg, double *__restrict__ g, double *err_part, int *status,
                   unsigned long long timeout_ns) {
    const long long j = (long long)blockIdx.x * 256 + threadIdx.x;
    double e2 = 0.0;
    if (j < D && *reinterpret_cast<volatile int *>(status) == 0) {
        const unsigned long long t0 = global_timer_ns();
        Lse acc{-INFINITY, 0.0};
        bool ok = true;
        for (int r = 0; r < G && ok; ++r) {
            const uint4 *src = ll_slot(ll_local, G, 2 * D, flag, r, 2 * j);
            unsigned long long m = 0, s = 0;
            ok = ll_poll(src, flag, m, t0, timeout_ns) && ll_poll(src + 1, flag, s, t0, timeout_ns);
            if (ok) lse_fold(acc, Lse{__longlong_as_double((long long)m), __longlong_as_double((long long)s)});
        }
        if (ok) e2 = sk_col_finish(acc, log_b[j], b[j], reg, g[j]);
        else atomicExch(status, SX_ERR_PEER_TIMEOUT);
    }
    const double t = sk_err_block_sum(e2);
    if (threadIdx.x == 0 && err_part != nullptr) err_part[blockIdx.x] = t;
}

__global__ void sk_log_kernel(const double *__restrict__ a, long long n, double *__restrict__ out) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        out[i] = log(a[i]);
}

__global__ void sk_fill_kernel(double *out, long long n, double v) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        out[i] = v;
}

// X_ij = exp((f_i + g_j - M_ij) / reg): a CTA per row (grid-stride), threads stride the columns.
__global__ void __launch_bounds__(256)
sk_plan_kernel(const double *__restrict__ M, long long ld, long long S, long long D, const double *__restrict__ f,
               const double *__restrict__ g, double reg, double *__restrict__ X) {
    const double inv = 1.0 / reg;
    for (long long i = blockIdx.x; i < S; i += gridDim.x) {
        const double fi = f[i];
        const double *row = M + i * ld;
        double *out = X + i * D;
        for (long long j = threadIdx.x; j < D; j += blockDim.x) out[j] = exp((fi + g[j] - __ldcs(row + j)) * inv);
    }
}

constexpr long long kSkRowsPerChunk = 128;

}  // namespace sx

using namespace sx;

extern "C" size_t sx_sinkhorn_workspace_bytes(int64_t S, int64_t D) {
    if (S < 0 || D < 0) return 0;
    const size_t chunks = ((size_t)S + kSkRowsPerChunk - 1) / kSkRowsPerChunk + 1;
    return carve_bytes((size_t)S, 8) + carve_bytes((size_t)D, 8) + 2 * carve_bytes(chunks * (size_t)D, 8) +
           carve_bytes(1, 8) + 256;
}

extern "C" int sx_sinkhorn_ot(const double *M, int64_t ld, int64_t S, int64_t D, const double *a, const double *b,
                              double reg, int64_t max_iter, double stop_thr, int64_t check_every, double *f,
                              double *g, double *x_out, int64_t *iters_h, double *err_h, void *ws, size_t ws_bytes,
                              void *stream) {
    if (!M || !a || !b || !f || !g || S <= 0 || D <= 0 || ld < D || !(reg > 0.0) || max_iter < 0) return SX_ERR_INVALID;
    if (!ws || ws_bytes < sx_sinkhorn_workspace_bytes(S, D)) return SX_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    if (check_every <= 0) check_every = 10;
    Carver cv(ws);
    double *log_a = cv.take<double>(S), *log_b = cv.take<double>(D);
    const long long n_chunks = (S + kSkRowsPerChunk - 1) / kSkRowsPerChunk;
    double *pm = cv.take<double>((size_t)n_chunks * D), *ps = cv.take<double>((size_t)n_chunks * D);
    double *err2 = cv.take<double>(1);
    sk_log_kernel<<<num_sms(), 256, 0, st>>>(a, S, log_a);
    sk_log_kernel<<<num_sms(), 256, 0, st>>>(b, D, log_b);
    SX_LAUNCH_CHECK();
    SX_CUDA(cudaMemsetAsync(g, 0, sizeof(double) * (size_t)D, st));
    sk_fill_kernel<<<num_sms(), 256, 0, st>>>(f, S, -reg * log((double)S));     // u = 1 / S
    SX_LAUNCH_CHECK();
    long long row_grid = (S * 32 + 255) / 256;
    if (row_grid > num_sms() * 16) row_grid = num_sms() * 16;
    const dim3 col_grid((unsigned)((D + 255) / 256), (unsigned)n_chunks);
    int64_t it = 0;
    double err = INFINITY;
    for (; it < max_iter; ++it) {
        // the column pass of iteration `it` also yields the marginal error of iteration it - 1
        const bool check = stop_thr > 0.0 && it > 0 && ((it - 1) % check_every == 0);
        if (check) SX_CUDA(cudaMemsetAsync(err2, 0, sizeof(double), st));
        sk_col_partial_kernel<<<col_grid, 256, 0, st>>>(M, ld, S, D, f, reg, kSkRowsPerChunk, pm, ps);
        SX_LAUNCH_CHECK();
        sk_col_merge_kernel<<<(int)((D + 255) / 256), 256, 0, st>>>(D, n_chunks, pm, ps, log_b, b, reg, g,
                                                                    check ? err2 : nullptr);
        SX_LAUNCH_CHECK();
        if (check) {
            double e2 = 0.0;
            SX_CUDA(cudaMemcpyAsync(&e2, err2, sizeof(double), cudaMemcpyDeviceToHost, st));
            SX_CUDA(cudaStreamSynchronize(st));
            err = sqrt(e2);
            if (err < stop_thr) break;
        }
        sk_row_kernel<<<(int)row_grid, 256, 0, st>>>(M, ld, S, D, g, log_a, reg, f);
        SX_LAUNCH_CHECK();
    }
    if (x_out) {
        sk_plan_kernel<<<num_sms() * 8, 256, 0, st>>>(M, ld, S, D, f, g, reg, x_out);
        SX_LAUNCH_CHECK();
    }
    if (iters_h) *iters_h = it;
    if (err_h) *err_h = err;
    return SX_OK;
}

namespace {

// Buffers of one rank of sx_sinkhorn_ot_sharded_h, carved from one allocation on the rank's device.
struct SkRank {
    int dev = 0;
    cudaStream_t st = nullptr;                 // the stream of this rank's device (ranks of one device share it)
    const double *M = nullptr;
    int64_t row0 = 0, S_loc = 0, n_chunks = 0;
    void *mem = nullptr;
    double *a = nullptr, *log_a = nullptr, *b = nullptr, *log_b = nullptr, *f = nullptr, *g = nullptr;
    double *pm = nullptr, *ps = nullptr;
    double *ctl = nullptr;                     // {status (int32), error part of each fold CTA}: one copy reads both
    char *ll_buf = nullptr;
    char **peer_bufs = nullptr;
    int *status() const { return reinterpret_cast<int *>(ctl); }
    double *err_part() const { return ctl + 1; }
};

struct SkSharded {
    std::vector<SkRank> r;
    std::vector<std::pair<int, cudaStream_t>> streams;   // one per distinct device
    int prev = 0;
    ~SkSharded() {
        for (auto &ds : streams) {
            cudaSetDevice(ds.first);
            cudaStreamSynchronize(ds.second);
            cudaStreamDestroy(ds.second);
        }
        for (SkRank &k : r) {
            if (!k.mem) continue;
            cudaSetDevice(k.dev);
            cudaFree(k.mem);
        }
        cudaSetDevice(prev);
    }
};

size_t sk_rank_bytes(int64_t S_loc, int64_t D, int64_t n_chunks, int G, unsigned col_blocks) {
    return 3 * carve_bytes((size_t)S_loc, 8) + 3 * carve_bytes((size_t)D, 8) +
           2 * carve_bytes((size_t)n_chunks * D, 8) + carve_bytes(1 + (size_t)col_blocks, 8) +
           carve_bytes((size_t)4 * G * D, 16) + carve_bytes((size_t)G, sizeof(void *));
}

}  // namespace

extern "C" int sx_sinkhorn_ot_sharded_h(int ndev, const int *devs, const double *const *slabs,
                                        const int64_t *row_bounds, int64_t ld, int64_t S, int64_t D,
                                        const double *a_h, const double *b_h, double reg, int64_t max_iter,
                                        double stop_thr, int64_t check_every, double *f_h, double *g_h,
                                        double *const *x_out, int64_t *iters_h, double *err_h) {
    if (ndev < 1 || ndev > 64 || !devs || !slabs || !a_h || !b_h || !f_h || !g_h || S < 1 || D < 1 || ld < D ||
        !(reg > 0.0) || max_iter < 0)
        return SX_ERR_INVALID;
    if (ndev > S) return SX_ERR_INVALID;                      // every rank needs at least one row
    if (row_bounds) {
        if (row_bounds[0] != 0 || row_bounds[ndev] != S) return SX_ERR_INVALID;
        for (int g = 0; g < ndev; ++g) if (row_bounds[g + 1] <= row_bounds[g]) return SX_ERR_INVALID;
    }
    for (int g = 0; g < ndev; ++g) if (!slabs[g] || (x_out && !x_out[g])) return SX_ERR_INVALID;
    if (check_every <= 0) check_every = 10;
    const int G = ndev;
    const unsigned col_blocks = (unsigned)((D + 255) / 256);
    SkSharded sh;
    SX_CUDA(cudaGetDevice(&sh.prev));
    sh.r.resize(G);
    for (int g = 0; g < G; ++g) {
        SkRank &k = sh.r[g];
        k.dev = devs[g];
        k.M = slabs[g];
        k.row0 = row_bounds ? row_bounds[g] : S * g / G;
        k.S_loc = (row_bounds ? row_bounds[g + 1] : S * (g + 1) / G) - k.row0;
        k.n_chunks = (k.S_loc + kSkRowsPerChunk - 1) / kSkRowsPerChunk;
        if (cudaSetDevice(k.dev) != cudaSuccess) return SX_ERR_NO_DEVICE;
        for (auto &ds : sh.streams) if (ds.first == k.dev) k.st = ds.second;
        if (!k.st) {                                          // first rank on this device
            int rc = enable_peer_access(k.dev, G, devs);
            if (rc != SX_OK) return rc;
            SX_CUDA(cudaStreamCreateWithFlags(&k.st, cudaStreamNonBlocking));
            sh.streams.emplace_back(k.dev, k.st);
        }
        const size_t bytes = sk_rank_bytes(k.S_loc, D, k.n_chunks, G, col_blocks);
        SX_CUDA(cudaMalloc(&k.mem, bytes));
        Carver cv(k.mem);
        k.a = cv.take<double>(k.S_loc); k.log_a = cv.take<double>(k.S_loc); k.f = cv.take<double>(k.S_loc);
        k.b = cv.take<double>(D); k.log_b = cv.take<double>(D); k.g = cv.take<double>(D);
        k.pm = cv.take<double>((size_t)k.n_chunks * D); k.ps = cv.take<double>((size_t)k.n_chunks * D);
        k.ctl = cv.take<double>(1 + (size_t)col_blocks);
        k.ll_buf = cv.take<char>((size_t)4 * G * D * 16);
        k.peer_bufs = cv.take<char *>(G);
        SX_CUDA(cudaMemsetAsync(k.ctl, 0, sizeof(double), k.st));
        SX_CUDA(cudaMemsetAsync(k.ll_buf, 0, (size_t)4 * G * D * 16, k.st));
        SX_CUDA(cudaMemcpyAsync(k.a, a_h + k.row0, (size_t)k.S_loc * 8, cudaMemcpyHostToDevice, k.st));
        SX_CUDA(cudaMemcpyAsync(k.b, b_h, (size_t)D * 8, cudaMemcpyHostToDevice, k.st));
        sk_log_kernel<<<num_sms(), 256, 0, k.st>>>(k.a, k.S_loc, k.log_a);
        sk_log_kernel<<<num_sms(), 256, 0, k.st>>>(k.b, D, k.log_b);
        SX_LAUNCH_CHECK();
        SX_CUDA(cudaMemsetAsync(k.g, 0, sizeof(double) * (size_t)D, k.st));
        sk_fill_kernel<<<num_sms(), 256, 0, k.st>>>(k.f, k.S_loc, -reg * log((double)S));     // u = 1 / S (global S)
        SX_LAUNCH_CHECK();
    }
    std::vector<char *> bufs(G);                              // every rank learns every exchange buffer
    for (int g = 0; g < G; ++g) bufs[g] = sh.r[g].ll_buf;
    for (SkRank &k : sh.r) {
        SX_CUDA(cudaSetDevice(k.dev));
        SX_CUDA(cudaMemcpyAsync(k.peer_bufs, bufs.data(), sizeof(void *) * G, cudaMemcpyHostToDevice, k.st));
    }
    for (auto &ds : sh.streams) {                             // buffers zeroed everywhere before any push
        SX_CUDA(cudaSetDevice(ds.first));
        SX_CUDA(cudaStreamSynchronize(ds.second));
    }
    const unsigned long long timeout_ns = 10ull * 1000 * 1000 * 1000;
    std::vector<double> ctl_h(1 + (size_t)col_blocks);
    SkRank &k0 = sh.r[0];
    int64_t it = 0;
    double err = INFINITY;
    // Enqueue order per iteration: partial + push of every rank, fold of every rank, row pass of every rank.  Ranks
    // that share a device share its stream, so there every push precedes every fold and no kernel waits on a later
    // one; ranks on distinct devices poll each other's pushes over NVLink.
    for (; it < max_iter; ++it) {
        const bool check = stop_thr > 0.0 && it > 0 && ((it - 1) % check_every == 0);
        const unsigned flag = (unsigned)(it + 1);
        for (int g = 0; g < G; ++g) {
            SkRank &k = sh.r[g];
            SX_CUDA(cudaSetDevice(k.dev));
            sk_col_partial_kernel<<<dim3(col_blocks, (unsigned)k.n_chunks), 256, 0, k.st>>>(
                k.M, ld, k.S_loc, D, k.f, reg, kSkRowsPerChunk, k.pm, k.ps);
            sk_col_push_kernel<<<col_blocks, 256, 0, k.st>>>(D, k.n_chunks, k.pm, k.ps, k.peer_bufs, g, G, flag);
            SX_LAUNCH_CHECK();
        }
        for (int g = 0; g < G; ++g) {
            SkRank &k = sh.r[g];
            SX_CUDA(cudaSetDevice(k.dev));
            sk_col_fold_kernel<<<col_blocks, 256, 0, k.st>>>(D, k.ll_buf, G, flag, k.log_b, k.b, reg, k.g,
                                                             (check && g == 0) ? k.err_part() : nullptr, k.status(),
                                                             timeout_ns);
            SX_LAUNCH_CHECK();
        }
        if (check) {                                          // rank 0's error decides for every rank
            SX_CUDA(cudaSetDevice(k0.dev));
            SX_CUDA(cudaMemcpyAsync(ctl_h.data(), k0.ctl, ctl_h.size() * 8, cudaMemcpyDeviceToHost, k0.st));
            SX_CUDA(cudaStreamSynchronize(k0.st));
            int status = 0;
            memcpy(&status, ctl_h.data(), sizeof(int));
            if (status != 0) return status;
            double e2 = 0.0;
            for (unsigned c = 0; c < col_blocks; ++c) e2 += ctl_h[1 + c];        // CTA order: deterministic
            err = sqrt(e2);
            if (err < stop_thr) break;
        }
        for (int g = 0; g < G; ++g) {
            SkRank &k = sh.r[g];
            SX_CUDA(cudaSetDevice(k.dev));
            long long row_grid = (k.S_loc * 32 + 255) / 256;
            if (row_grid > num_sms() * 16) row_grid = num_sms() * 16;
            sk_row_kernel<<<(int)row_grid, 256, 0, k.st>>>(k.M, ld, k.S_loc, D, k.g, k.log_a, reg, k.f);
            SX_LAUNCH_CHECK();
        }
    }
    int status = SX_OK;
    for (int g = 0; g < G; ++g) {
        SkRank &k = sh.r[g];
        SX_CUDA(cudaSetDevice(k.dev));
        if (x_out) {
            sk_plan_kernel<<<num_sms() * 8, 256, 0, k.st>>>(k.M, ld, k.S_loc, D, k.f, k.g, reg, x_out[g]);
            SX_LAUNCH_CHECK();
        }
        SX_CUDA(cudaMemcpyAsync(f_h + k.row0, k.f, (size_t)k.S_loc * 8, cudaMemcpyDeviceToHost, k.st));
        if (g == 0) SX_CUDA(cudaMemcpyAsync(g_h, k.g, (size_t)D * 8, cudaMemcpyDeviceToHost, k.st));
        int s = 0;
        SX_CUDA(cudaMemcpyAsync(&s, k.status(), sizeof(int), cudaMemcpyDeviceToHost, k.st));
        SX_CUDA(cudaStreamSynchronize(k.st));
        if (status == SX_OK) status = s;
    }
    if (status != SX_OK) return status;
    if (iters_h) *iters_h = it;
    if (err_h) *err_h = err;
    return SX_OK;
}

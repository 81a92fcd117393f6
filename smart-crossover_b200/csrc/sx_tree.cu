// sx_tree.cu -- K3: node potentials of a spanning tree by Euler tour + list ranking (sm_100a).
//
// The reference takes the duals from the LP solver (`return_y`, solver_caller/gurobi.py:157-159,
// consumed at network_methods/algorithms.py:132).  For a tree basis they are the solution of
// B^T y[:-1] = c[tree], y[root] = 0 with B = A[:-1, tree] (tree_BI.py:74): every tree arc fixes
// y[plus] - y[minus] = cost.  Here:
//   1. every tree arc becomes two half-edges (minus->plus carrying +c, plus->minus carrying -c);
//   2. half-edges are sorted by origin node (radix argsort) to get each node's adjacency;
//   3. succ(u->v) = the half-edge after (v->u) in v's circular adjacency list = Euler tour;
//      the tour is cut at the root's first half-edge;
//   4. Wyllie pointer jumping over `pred` accumulates, for every half-edge, the inclusive prefix
//      of the weights (fp64) and of ones (its position in the tour) in ceil(log2 2T) rounds;
//   5. of each pair of half-edges the one met first goes down the tree, and the prefix sum at
//      it is the potential of the node it enters.
// Latency / L2-gather bound (2T <= 2.4e5 elements at C5).
//
// The same tour gives the tree's primal flows (sx_tree_flows; reference tree_BI.py:74-76 solves
// B x = b[:-1] with SuperLU): the flow on a tree arc is +/- the sum of the supplies b over the
// subtree hanging below it, i.e. a difference of two prefix sums of b taken in tour order.  The
// prefix sums are carried in double-double (error-free TwoSum): each prefix is off by at most about
// 2^-105 H sum|b| (sum over the non-root nodes), so a flow is within 1/2 ulp + 2^-103 H sum|b| of the
// exact subtree sum s, which is within 1 ulp of s whenever sum|b| <= 2^50 |s| / H.  It is not 1 ulp
// regardless of the running total: a subtree sum 1e20 times smaller than sum|b| loses digits.
//
// Accuracy of the potentials (plain fp64 sums): every partial sum of the pointer jumping is the sum of
// a contiguous stretch of the tour, i.e. a difference of two potentials.  So the potentials are exact
// when all costs are multiples of one 2^-e and max|y| < 2^52 * 2^-e (integer costs, for one), and in
// general the error is normwise, under one eps * max|y| per round: tested at <= 2 ceil(log2 H) eps max|y|.
// Relative to a node's own |y| it can be far larger: with 1% of the costs 1e6 times the rest, tens of
// thousands of nodes of a 1e5-node tree miss 1e-9 * |y| (DESIGN.md, tree kernels against exact references).
#include "sx_common.cuh"
#include "sx_gridbar.cuh"

namespace sx {

constexpr int kTrThreads = 256;
constexpr int kTourThreads = 1024;     // the cooperative tour kernel: few, fat CTAs make the grid barrier cheap
constexpr long long kTourSmallH = 4096; // up to here one CTA ranks the whole tour in shared memory (128 KB)

// Ranking state of a half-edge: inclusive prefix of the weights, tour position, predecessor still to jump over.
// One 16-byte record: a pointer-jumping round is two 128-bit gathers per element instead of six loads.
struct __align__(16) TourNode {
    double sum;
    int    rank;
    int    pred;
};

struct TreeArrays {
    unsigned long long *origin;   // H sort keys: origin node of each half-edge
    unsigned long long *sorted_origin;   // H
    uint32_t *ho;                 // H half-edge ids sorted by origin (stable)
    int      *dest;               // H
    int      *pos;                // H position of a half-edge in `ho`
    int      *first;              // N first position of a node's run in `ho`, -1 if none
    TourNode *node[2];            // H, ping-pong of the pointer jumping
};

__global__ void tree_halfedges_kernel(const long long *__restrict__ tree, long long T,
                                      const int32_t *__restrict__ tail, const int32_t *__restrict__ head,
                                      long long S, long long D, const double *__restrict__ cost, long long ld,
                                      int plus_is_tail, TreeArrays a) {
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < T;
         t += (long long)gridDim.x * blockDim.x) {
        const long long e = tree[t];
        int plus, minus;
        double c;
        if (tail == nullptr) {
            const long long i = e / D, j = e - i * D;
            plus = (int)(S + j); minus = (int)i;
            c = cost ? cost[i * ld + j] : 0.0;
        } else {
            plus = plus_is_tail ? tail[e] : head[e];
            minus = plus_is_tail ? head[e] : tail[e];
            c = cost ? cost[e] : 0.0;
        }
        a.origin[2 * t] = (unsigned long long)minus; a.dest[2 * t] = plus;      a.node[0][2 * t].sum = c;
        a.origin[2 * t + 1] = (unsigned long long)plus; a.dest[2 * t + 1] = minus; a.node[0][2 * t + 1].sum = -c;
    }
}

__device__ __forceinline__ TourNode ld_node(const TourNode *p) {
    const int4 v = __ldcg(reinterpret_cast<const int4 *>(p));
    TourNode n;
    n.sum = __hiloint2double(v.y, v.x); n.rank = v.z; n.pred = v.w;
    return n;
}

// Everything between the half-edge sort and the read-out in ONE launch: adjacency (first / pos), Euler
// successor, cut at the root, and the ceil(log2 H) pointer-jumping rounds, separated by barriers instead of
// kernel boundaries -- 17-21 launches of ~5 us each used to be most of the potentials' time.  Large tours run
// cooperatively (grid-wide barriers, sx_gridbar.cuh; the grid is sized to the work); a tour of up to
// kTourSmallH half-edges is ranked by ONE CTA with the ping-pong records in shared memory and __syncthreads
// as the barrier.  Leaves the result in node[rounds & 1].
__global__ void __launch_bounds__(kTourThreads)
tree_tour_kernel(long long H, long long N, long long root, int rounds, TreeArrays a, GridBarrier *bar, int32_t *status) {
    extern __shared__ __align__(16) unsigned char tour_raw[];
    const bool single = gridDim.x == 1;
    auto sync_all = [&]() { if (single) __syncthreads(); else grid_barrier(bar); };
    const long long gtid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long gsz = (long long)gridDim.x * blockDim.x;
    for (long long v = gtid; v <= N; v += gsz) a.first[v] = -1;
    sync_all();
    for (long long p = gtid; p < H; p += gsz) {
        const unsigned long long v = a.sorted_origin[p];
        if (p == 0 || a.sorted_origin[p - 1] != v) a.first[v] = (int)p;
        a.pos[a.ho[p]] = (int)p;
    }
    sync_all();
    for (long long h = gtid; h < H; h += gsz) {
        const long long twin = h ^ 1;
        const unsigned long long v = (unsigned long long)a.dest[h];
        long long p2 = (long long)__ldcg(a.pos + twin) + 1;
        if (p2 >= H || a.sorted_origin[p2] != v) p2 = __ldcg(a.first + v);
        const uint32_t succ = a.ho[p2];
        a.node[0][succ].pred = (int)h;
        a.node[0][h].rank = 1;
    }
    // A node without a half-edge is not spanned.  This check is needed as well as the one on unreached
    // half-edges in the read-out: N - 1 arcs with a cycle can still form ONE tour through every half-edge
    // (three parallel arcs between two nodes do), and then only the isolated nodes give them away.
    for (long long v = gtid; v < N; v += gsz)
        if (__ldcg(a.first + v) < 0) *status = SX_ERR_NOT_SPANNING;
    sync_all();
    if (gtid == 0) {
        const int f = __ldcg(a.first + root);
        if (f < 0) *status = SX_ERR_NOT_SPANNING; else a.node[0][a.ho[f]].pred = -1;
    }
    sync_all();
    if (single && H <= kTourSmallH) {
        TourNode *in = reinterpret_cast<TourNode *>(tour_raw), *out = in + H;
        for (long long h = threadIdx.x; h < H; h += blockDim.x) in[h] = ld_node(a.node[0] + h);
        __syncthreads();
        for (int r = 0; r < rounds; ++r) {
            for (long long h = threadIdx.x; h < H; h += blockDim.x) {
                TourNode me = in[h];
                if (me.pred >= 0) {
                    const TourNode pr = in[me.pred];
                    me.sum = pr.sum + me.sum; me.rank += pr.rank; me.pred = pr.pred;
                }
                out[h] = me;
            }
            __syncthreads();
            TourNode *t = in; in = out; out = t;
        }
        TourNode *res = (rounds & 1) ? a.node[1] : a.node[0];
        for (long long h = threadIdx.x; h < H; h += blockDim.x) res[h] = in[h];
        return;
    }
    const TourNode *in = a.node[0];
    TourNode *out = a.node[1];
    for (int r = 0; r < rounds; ++r) {
        for (long long h = gtid; h < H; h += gsz) {
            TourNode me = ld_node(in + h);
            if (me.pred >= 0) {
                const TourNode pr = ld_node(in + me.pred);
                me.sum = pr.sum + me.sum; me.rank += pr.rank; me.pred = pr.pred;
            }
            out[h] = me;
        }
        sync_all();
        TourNode *t = const_cast<TourNode *>(in); in = out; out = t;
    }
}

__global__ void tree_finalize_kernel(long long T, long long root, const TourNode *__restrict__ node,
                                     const int *__restrict__ dest, double *__restrict__ y, int32_t *status) {
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < T;
         t += (long long)gridDim.x * blockDim.x) {
        const long long ha = 2 * t, hb = 2 * t + 1;
        const TourNode na = node[ha], nb = node[hb];
        if (na.pred != -1 || nb.pred != -1) { *status = SX_ERR_NOT_SPANNING; continue; }
        y[dest[na.rank < nb.rank ? ha : hb]] = na.rank < nb.rank ? na.sum : nb.sum;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) y[root] = 0.0;
}

__global__ void tree_status_kernel(int32_t *status, int32_t v) { *status = v; }

// ---- primal flows ------------------------------------------------------------------------
struct dd { double hi, lo; };
__device__ __forceinline__ dd dd_add(dd a, double b) {           // error-free a + b (Knuth TwoSum), renormalised
    const double s = a.hi + b;
    const double bb = s - a.hi;
    const double e = (a.hi - (s - bb)) + (b - bb);
    const double lo = a.lo + e;
    const double hi = s + lo;
    return dd{hi, lo - (hi - s)};
}
__device__ __forceinline__ dd dd_add(dd a, dd b) { return dd_add(dd_add(a, b.hi), b.lo); }

// w[pos] = supply of the node entered at tour position pos (down half-edges), 0 for up half-edges.
__global__ void flow_scatter_kernel(long long T, const TourNode *__restrict__ node,
                                    const int *__restrict__ dest, const double *__restrict__ b, double *__restrict__ w,
                                    int32_t *status) {
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < T;
         t += (long long)gridDim.x * blockDim.x) {
        const long long ha = 2 * t, hb = 2 * t + 1;
        const TourNode na = node[ha], nb = node[hb];
        if (na.pred != -1 || nb.pred != -1) { *status = SX_ERR_NOT_SPANNING; continue; }
        const bool a_down = na.rank < nb.rank;
        const long long down = a_down ? ha : hb;
        w[(a_down ? na.rank : nb.rank) - 1] = b[dest[down]];
        w[(a_down ? nb.rank : na.rank) - 1] = 0.0;
    }
}

// One CTA: inclusive double-double prefix sum of w[0..H) -> (phi, plo).
__global__ void __launch_bounds__(1024) flow_scan_kernel(long long H, const double *__restrict__ w,
                                                         double *__restrict__ phi, double *__restrict__ plo) {
    __shared__ double s_hi[1024], s_lo[1024];
    const long long chunk = (H + 1023) / 1024;
    const long long lo = (long long)threadIdx.x * chunk, hi = lo + chunk < H ? lo + chunk : H;
    dd acc{0.0, 0.0};
    for (long long i = lo; i < hi; ++i) acc = dd_add(acc, w[i]);
    s_hi[threadIdx.x] = acc.hi; s_lo[threadIdx.x] = acc.lo;
    __syncthreads();
    if (threadIdx.x == 0) {                                     // 1024 chunk totals: serial exclusive scan
        dd run{0.0, 0.0};
        for (int i = 0; i < 1024; ++i) {
            const dd v{s_hi[i], s_lo[i]};
            s_hi[i] = run.hi; s_lo[i] = run.lo;
            run = dd_add(run, v);
        }
    }
    __syncthreads();
    acc = dd{s_hi[threadIdx.x], s_lo[threadIdx.x]};
    for (long long i = lo; i < hi; ++i) {
        acc = dd_add(acc, w[i]);
        phi[i] = acc.hi; plo[i] = acc.lo;
    }
}

// flow(t) = +/- (P[rank(up) - 1] - P[rank(down) - 2]): supplies of the subtree below arc t.
// Arcs the tour never reached (not spanning; flow_scatter_kernel has set the status) are skipped: their
// ranks run up to 2^rounds, past the H prefix sums.
__global__ void flow_finalize_kernel(long long T, const TourNode *__restrict__ node,
                                     const double *__restrict__ phi, const double *__restrict__ plo,
                                     double *__restrict__ flow) {
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < T;
         t += (long long)gridDim.x * blockDim.x) {
        const long long ha = 2 * t, hb = 2 * t + 1;            // ha: minus -> plus, hb: plus -> minus
        const TourNode na = node[ha], nb = node[hb];
        if (na.pred != -1 || nb.pred != -1) continue;
        const int ra = na.rank, rb = nb.rank;
        const bool a_down = ra < rb;
        const long long r1 = (a_down ? ra : rb) - 1, r2 = (a_down ? rb : ra) - 1;  // tour positions (down, up), r1 < r2
        dd top{phi[r2], plo[r2]};
        if (r1 > 0) top = dd_add(top, dd{-phi[r1 - 1], -plo[r1 - 1]});
        const double subtree = top.hi + top.lo;
        // the arc's column has +1 at `plus`, -1 at `minus`; conservation over the subtree gives the sign
        flow[t] = a_down ? subtree : -subtree;
    }
}

static int tr_grid(long long n) {
    long long g = (n + kTrThreads - 1) / kTrThreads;
    if (g > num_sms() * 8) g = num_sms() * 8;
    if (g < 1) g = 1;
    return (int)g;
}

}  // namespace sx

using namespace sx;

extern "C" size_t sx_tree_potentials_workspace_bytes(int64_t N) {
    if (N < 0) return 0;
    const size_t H = 2 * (size_t)(N > 0 ? N : 1);
    return 2 * carve_bytes(H, 8) + carve_bytes(H, 4) * 3 + carve_bytes((size_t)N + 1, 4) +
           2 * carve_bytes(H, 16) + sx_argsort_workspace_bytes((int64_t)H) + 1024;
}

// Shared by potentials and flows: half-edges, Euler tour cut at the root, pointer jumping.
// On return a.sum[cur] / a.rank[cur] / a.pred[cur] hold the inclusive prefix of the half-edge
// weights, the 1-based tour position, and -1 for every half-edge reached from the root.
static int tree_tour(const int64_t *tree, int64_t n_tree, const int32_t *tail, const int32_t *head, int64_t S,
                     int64_t D, int64_t N, const double *cost, int64_t ld, int plus_convention, int64_t root,
                     int32_t *status_out, void *ws, size_t ws_bytes, cudaStream_t st, TreeArrays &a, int &cur) {
    const long long T = n_tree, H = 2 * T;
    Carver cv(ws);
    a.origin = cv.take<unsigned long long>(H);
    a.sorted_origin = cv.take<unsigned long long>(H);
    a.ho = cv.take<uint32_t>(H);
    a.dest = cv.take<int>(H);
    a.pos = cv.take<int>(H);
    a.first = cv.take<int>(N + 1);
    a.node[0] = cv.take<TourNode>(H); a.node[1] = cv.take<TourNode>(H);
    GridBarrier *bar = cv.take<GridBarrier>(1);
    void *sort_ws = cv.base + cv.off;
    const size_t sort_ws_bytes = ws_bytes - cv.off;

    tree_halfedges_kernel<<<tr_grid(T), kTrThreads, 0, st>>>((const long long *)tree, T, tail, head, S, D, cost, ld,
                                                             plus_convention == SX_PLUS_IS_TAIL, a);
    SX_LAUNCH_CHECK();
    int bits = 1;
    while (bits < 32 && (1ll << bits) < N) ++bits;
    int rc = sx_argsort_u64(a.origin, H, bits, a.ho, a.sorted_origin, sort_ws, sort_ws_bytes, st);
    if (rc != SX_OK) return rc;
    int rounds = 1;
    while ((1ll << rounds) < H) ++rounds;
    cur = rounds & 1;
    SX_CUDA(cudaMemsetAsync(bar, 0, sizeof(GridBarrier), st));
    long long H_ = H, N_ = N, root_ = root;
    void *args[] = {(void *)&H_, (void *)&N_, (void *)&root_, (void *)&rounds, (void *)&a, (void *)&bar, (void *)&status_out};
    if (H <= kTourSmallH) {
        const size_t smem = (size_t)2 * H * sizeof(TourNode);
        SX_CUDA(cudaFuncSetAttribute(tree_tour_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)(2 * kTourSmallH * sizeof(TourNode))));
        SX_CUDA(cudaLaunchKernel((void *)tree_tour_kernel, dim3(1), dim3(kTourThreads), args, smem, st));
    } else {
        int occ = 0;
        SX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, tree_tour_kernel, kTourThreads, 0));
        if (occ < 1) return SX_ERR_NO_DEVICE;
        long long grid = (H + kTourThreads - 1) / kTourThreads;
        const long long max_grid = (long long)num_sms() * (occ > 2 ? 2 : occ);
        if (grid > max_grid) grid = max_grid;
        SX_CUDA(cudaLaunchCooperativeKernel((void *)tree_tour_kernel, dim3((unsigned)grid), dim3(kTourThreads), args, 0, st));
    }
    return SX_OK;
}

static int tree_check_args(const void *out, const int32_t *status_out, const int32_t *tail, const int32_t *head,
                           int64_t S, int64_t D, int64_t N, int64_t ld, int64_t root, int64_t n_tree, const void *ws,
                           size_t ws_bytes) {
    if (!out || !status_out || N <= 0 || root < 0 || root >= N || n_tree < 0) return SX_ERR_INVALID;
    if ((tail == nullptr) != (head == nullptr)) return SX_ERR_INVALID;
    if (!tail && (S <= 0 || D <= 0 || S + D != N || ld < D)) return SX_ERR_INVALID;
    if (N >= (1ll << 30)) return SX_ERR_TOO_LARGE;
    if (!ws || ws_bytes < sx_tree_potentials_workspace_bytes(N)) return SX_ERR_WORKSPACE;
    return SX_OK;
}

extern "C" int sx_tree_potentials(const int64_t *tree, int64_t n_tree, const int32_t *tail, const int32_t *head,
                                  int64_t S, int64_t D, int64_t N, const double *cost, int64_t ld,
                                  int plus_convention, int64_t root, double *y_out, int32_t *status_out,
                                  void *ws, size_t ws_bytes, void *stream) {
    int arg = tree_check_args(y_out, status_out, tail, head, S, D, N, ld, root, n_tree, ws, ws_bytes);
    if (arg != SX_OK) return arg;
    cudaStream_t st = (cudaStream_t)stream;
    if (n_tree != N - 1) {   // cannot be a spanning tree
        tree_status_kernel<<<1, 1, 0, st>>>(status_out, SX_ERR_NOT_SPANNING);
        SX_LAUNCH_CHECK();
        return SX_OK;
    }
    tree_status_kernel<<<1, 1, 0, st>>>(status_out, 0);
    SX_LAUNCH_CHECK();
    if (N == 1) {
        SX_CUDA(cudaMemsetAsync(y_out, 0, sizeof(double), st));
        return SX_OK;
    }
    if (!tree || !cost) return SX_ERR_INVALID;
    TreeArrays a;
    int cur = 0;
    int rc = tree_tour(tree, n_tree, tail, head, S, D, N, cost, ld, plus_convention, root, status_out, ws, ws_bytes, st,
                       a, cur);
    if (rc != SX_OK) return rc;
    tree_finalize_kernel<<<tr_grid(n_tree), kTrThreads, 0, st>>>(n_tree, root, a.node[cur], a.dest, y_out, status_out);
    SX_LAUNCH_CHECK();
    return SX_OK;
}

extern "C" int sx_tree_flows(const int64_t *tree, int64_t n_tree, const int32_t *tail, const int32_t *head,
                             int64_t S, int64_t D, int64_t N, const double *b, int plus_convention, int64_t root,
                             double *flow_out, int32_t *status_out, void *ws, size_t ws_bytes, void *stream) {
    int arg = tree_check_args(flow_out, status_out, tail, head, S, D, N, D, root, n_tree, ws, ws_bytes);
    if (arg != SX_OK) return arg;
    cudaStream_t st = (cudaStream_t)stream;
    if (n_tree != N - 1) {
        tree_status_kernel<<<1, 1, 0, st>>>(status_out, SX_ERR_NOT_SPANNING);
        SX_LAUNCH_CHECK();
        return SX_OK;
    }
    tree_status_kernel<<<1, 1, 0, st>>>(status_out, 0);
    SX_LAUNCH_CHECK();
    if (N == 1) return SX_OK;
    if (!tree || !b) return SX_ERR_INVALID;
    TreeArrays a;
    int cur = 0;
    // the tour does not depend on the half-edge weights: b stands in for the cost array (one value per
    // arc is read for OT through cost[i * ld + j] with ld = D, which b does not have) -> use a zero-cost view
    int rc = tree_tour(tree, n_tree, tail, head, S, D, N, nullptr, D, plus_convention, root, status_out, ws, ws_bytes,
                       st, a, cur);
    if (rc != SX_OK) return rc;
    const long long T = n_tree, H = 2 * T;
    // scratch: the buffers of the finished ranking that are no longer needed
    double *w = reinterpret_cast<double *>(a.node[cur ^ 1]);
    double *phi = reinterpret_cast<double *>(a.origin), *plo = reinterpret_cast<double *>(a.sorted_origin);
    flow_scatter_kernel<<<tr_grid(T), kTrThreads, 0, st>>>(T, a.node[cur], a.dest, b, w, status_out);
    SX_LAUNCH_CHECK();
    flow_scan_kernel<<<1, 1024, 0, st>>>(H, w, phi, plo);
    SX_LAUNCH_CHECK();
    flow_finalize_kernel<<<tr_grid(T), kTrThreads, 0, st>>>(T, a.node[cur], phi, plo, flow_out);
    SX_LAUNCH_CHECK();
    return SX_OK;
}

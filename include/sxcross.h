/*
 * sxcross.h -- C ABI of libsxcross, the B200 (sm_100a) network-crossover hot path.
 *
 * This is the drop-in boundary.  The reference (wcwj0147/smart-crossover) is pure
 * Python; the arithmetic of its hot path runs inside NumPy / SciPy calls made from
 * `smart_crossover/network_methods/{net_manager,tree_BI,algorithms}.py`.  Each entry
 * point below replaces one of those call sites (cited as file:line relative to
 * /root/reference/src/smart_crossover/) and is what a ctypes binding inside the
 * reference's managers would bind (see INTEGRATION.md).
 *
 * Conventions
 *  - extern "C", plain pointers and sizes; no C++ or torch types.
 *  - Every function returns 0 (SX_OK) or a negative SX_ERR_* code; nothing throws.
 *  - Pointers are DEVICE pointers owned by the caller unless the parameter name ends
 *    in `_h` (host pointer).  No hidden allocation: `sx_*_workspace_bytes` reports the
 *    scratch a call needs and the caller passes `ws` / `ws_bytes`.  The one exception is
 *    the opaque handle sx_ot_pricer, which owns its buffers from create to destroy.
 *  - No per-call state lives in the library.  The `sx_*_set_tuning` functions set
 *    PROCESS-WIDE defaults (kernel shapes) for bench sweeps and tests; the product path
 *    never calls them and they are not meant to be changed while another thread is
 *    inside the library.
 *  - `stream` is a cudaStream_t passed as void*; calls are asynchronous with respect
 *    to the host and ordered by that stream, except the `_h` entry points, which
 *    synchronise the stream before returning.
 *  - Reals are IEEE fp64, computed without fast-math or FMA contraction.  Arc ids are
 *    uint32 inside the sort (n < 2^32) and int64 at the boundary.
 *  - OT arc id k = i * D + j; OT nodes: sources 0..S-1, sinks S..S+D-1
 *    (formats.py:156-160, net_manager.py:366).  Arc lists use tail/head int32 arrays.
 */
#ifndef SXCROSS_H_
#define SXCROSS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define SX_API __attribute__((visibility("default")))
#else
#define SX_API
#endif

#define SX_OK                   0
#define SX_ERR_INVALID         -1   /* bad argument (null pointer, negative size, ...) */
#define SX_ERR_CUDA            -2   /* a CUDA runtime call failed; see sx_last_cuda_error() */
#define SX_ERR_WORKSPACE       -3   /* ws_bytes smaller than sx_*_workspace_bytes() */
#define SX_ERR_TOO_LARGE       -4   /* n >= 2^32 arcs in a sort, or N >= 2^31 nodes */
#define SX_ERR_NOT_SPANNING    -5   /* sx_tree_potentials: arcs are not a spanning tree */
#define SX_ERR_UNALIGNED       -6   /* TMA path needs 16-byte aligned base and even ld */
#define SX_ERR_NO_DEVICE       -7   /* no sm_100 device / driver entry point missing */
#define SX_ERR_PEER_TIMEOUT    -8   /* sx_exchange_blocks: a peer never raised its flag */
#define SX_ERR_PUSH_ASSERT     -9   /* sx_push_tree_h: the reference's assertions would fire (tree_BI.py:93-94) */

#define SX_ABI_VERSION 6

/* Endpoint convention of sx_tree_potentials (which end of an arc carries +1 in A). */
#define SX_PLUS_IS_HEAD 0   /* OT:  A[S+j,k] = +1, A[i,k] = -1      (formats.py:156-158)     */
#define SX_PLUS_IS_TAIL 1   /* MCF: A[tail,k] = +1, A[head,k] = -1  (scripts/min2mcf.py:36-37) */

/* Result header of a pricing pass (device memory, 32 bytes, written by sx_price_*). */
typedef struct sx_price_header {
    unsigned long long n_violating;   /* #arcs with rc < -tol (exact, even past the candidate cap) */
    long long          min_rc_key;    /* order-preserving int64 image of min rc; see sx_key_to_f64 */
    unsigned long long n_priced;      /* arcs priced by this launch (sanity / throughput) */
    unsigned long long status;        /* SX_STATUS_* bits; 0 = the selection below is complete */
} sx_price_header;

#define SX_STATUS_CAND_OVERFLOW  1   /* candidate buffer too small: enlarge it and price again */
#define SX_STATUS_DUPLICATE_CANDIDATES 2   /* the candidates repeat one (rc, id) pair too often to select
                                              from: the same arcs were priced into one pass more than once.
                                              The selection is void; no repeat can fix it */
#define SX_STATUS_K_MISMATCH     4   /* sx_topk_select asked for more arcs than sx_price_pass_begin
                                        announced: the candidates were pruned for the smaller K */
#define SX_STATUS_NAN_RC         8   /* some reduced cost was NaN.  It is neither counted in n_violating nor
                                        selected (NumPy: NaN < -tol is False), but the optimality test
                                        `np.all(rc >= -tol)` (net_manager.py:318,496) is False: callers must
                                        treat the pass as NOT optimal.  Informational, no repeat needed. */
#define SX_STATUS_REPEAT_MASK    1   /* bits that ask for the pass to be repeated */

/* Selection state of a pricing pass (opaque device memory, sx_select_state_bytes() bytes, 16 B
 * aligned): candidate counter, pruning bound and the reduced-cost histogram the bound is derived
 * from.  Zeroed by sx_price_pass_begin, filled by sx_price_*, consumed by sx_topk_select. */
typedef struct sx_select_state sx_select_state;

SX_API int         sx_abi_version(void);
SX_API const char *sx_error_string(int code);
SX_API int         sx_last_cuda_error(void);            /* cudaError_t of the last SX_ERR_CUDA */
SX_API double      sx_key_to_f64(long long key);        /* decode sx_price_header.min_rc_key */

/* ---- K1: flow indicators ------------------------------------------------------------
 * sx_score_ot replaces `np.maximum(X / s[:,None], X / d[None,:])`, net_manager.py:377-378.
 *   x (S*D), s (S), d (D) -> score_out (S*D).  Correctly rounded IEEE divisions; NumPy
 *   `maximum` semantics (NaN propagates).  hist12_out (may be NULL; 4096 uint32, zeroed by the
 *   caller): histogram of the scores' top 12 key bits, accumulated while the scores are written,
 *   which sx_kruskal_prefix and sx_order_head_sharded_h accept instead of taking it with a pass of their own.
 * sx_score_mcf replaces net_manager.py:165-182: reversal of arcs with x > u/2, per-node
 *   out/in sums in ascending arc id (SciPy csr_matvec order), f_inv = 1/max(f1,f2),
 *   indicator = max over the two end nodes of |f_inv * x_hat|.  node_ptr (N+1) /
 *   node_arc / node_sign are the CSR arrays of the incidence matrix A (formats.py:118).
 *   An entry with node_sign 0 (a stored zero of A) is no incidence: it enters neither sum, so a
 *   NaN or infinite x_hat cannot reach that node through it.  u = inf gives x_hat = x + inf * 0 =
 *   NaN, as in the reference; f = inf gives f_inv = 0, a subnormal f gives f_inv = inf.
 */
SX_API int    sx_score_ot(const double *x, const double *s, const double *d, int64_t S, int64_t D,
                   double *score_out, uint32_t *hist12_out, void *stream);
SX_API int    sx_score_set_tuning(int min_ctas_per_sm);   /* 4 (default, 64 registers) or 3 (78 registers) resident CTAs per SM,
                                                             anything else SX_ERR_INVALID.  Both return the same scores and
                                                             histogram bits; process-wide, for bench sweeps */
SX_API size_t sx_score_mcf_workspace_bytes(int64_t N, int64_t E);
SX_API int    sx_score_mcf(const double *x, const double *u, const int32_t *tail, const int32_t *head,
                    const int64_t *node_ptr, const int32_t *node_arc, const int8_t *node_sign,
                    int64_t N, int64_t E, double *score_out, void *ws, size_t ws_bytes,
                    void *stream);

/* ---- K1c: stable radix argsort --------------------------------------------------------
 * Replaces `np.argsort(flow_indicators)` at net_manager.py:184,379 (run stable, north_star)
 * and the stable argsort inside scipy.sparse.csgraph.minimum_spanning_tree (tree_BI.py:53).
 *   order_asc_out[p] = arc id of the p-th smallest key; ties by ascending arc id;
 *   -0.0 == +0.0; NaN sorts last (NumPy order).  sorted_key_out (optional, may be NULL)
 *   receives the keys in sorted order.
 * sx_argsort_u64: the same order for uint64 keys, by their low 8 * max(2, ceil(key_bits / 8)) bits
 *   (1 <= key_bits <= 64): whole bytes, at least two, so key_bits <= 16 sorts 16 bits and 17 sorts 24.
 *   Bits above that range do not enter the order (keys equal below it are ties, by ascending id) and the
 *   keys need not be below 2^key_bits; sorted_key_out carries each key whole, those bits included.
 * sx_queue_from_order:   queue = order_asc[::-1] widened to int64 (net_manager.py:184,379).
 * sx_kruskal_order:      descending key, ties by ASCENDING id = stable argsort of -key, the
 *   order SciPy's Kruskal visits arcs in (tree_BI.py:47,53; SURVEY.md H1).
 */
SX_API int    sx_sort_set_tuning(int downsweep_threads);   /* 256, 384, 512 or 1024 threads per tile of the large-input
                                                              downsweep, 2 = chosen by size (default: 1024 from 2^26 keys); 0 / 1: mid-size inputs as launches per pass / as ONE
                                                              cooperative launch (default).  Process-wide, for bench sweeps */
SX_API size_t sx_argsort_workspace_bytes(int64_t n);
SX_API int    sx_argsort_f64(const double *key, int64_t n, uint32_t *order_asc_out,
                      double *sorted_key_out, void *ws, size_t ws_bytes, void *stream);
SX_API int    sx_argsort_u64(const unsigned long long *key, int64_t n, int key_bits,
                      uint32_t *order_asc_out, unsigned long long *sorted_key_out,
                      void *ws, size_t ws_bytes, void *stream);
SX_API int    sx_queue_from_order(const uint32_t *order_asc, int64_t n, int64_t *queue_out, void *stream);
SX_API size_t sx_kruskal_order_workspace_bytes(int64_t n);
SX_API int    sx_kruskal_order(const double *sorted_key, const uint32_t *order_asc, int64_t n,
                        uint32_t *korder_out, void *ws, size_t ws_bytes, void *stream);
/* Head of that order when only the heaviest arcs are needed (the tree build reads ~8 N of them): the tie
 * runs covering the last T ascending positions, flipped.  *n_head_h (HOST) = arcs written (>= T), or -1 when
 * the runs hold more than T_cap arcs (flip everything instead).  ws: sx_kruskal_order_workspace_bytes(T_cap)
 * + 256 bytes.  One stream synchronisation. */
SX_API int    sx_kruskal_order_head(const double *sorted_key, const uint32_t *order_asc, int64_t n, int64_t T,
                             int64_t T_cap, uint32_t *korder_out, int64_t *n_head_h, void *ws,
                             size_t ws_bytes, void *stream);

/* ---- K1d: head of the Kruskal order without a full sort ---------------------------------
 * `max_weight_spanning_tree` (tree_BI.py:32-59) passes all n weights to SciPy's Kruskal, which
 * argsorts them all although the tree is complete after the first few N arcs.  sx_kruskal_prefix
 * returns only the head of that order: every arc whose weight is >= the T-th largest one (to 24
 * bits of its order-preserving image), in Kruskal order (descending weight, ties by ascending
 * arc id), i.e. exactly the first *n_prefix_h entries of what sx_argsort_f64 + sx_kruskal_order
 * would produce.  One to three streaming passes over the weights (8-24 B per arc: the top-12-bit
 * histogram unless the caller has it, one split pass, and two more passes only when the threshold
 * bin is too crowded for the boundary list) instead of ~256 B per arc.
 *   hist12 (may be NULL): the 4096-bin histogram of the weights' top 12 key bits if the caller has
 *   it already (sx_score_ot / sx_hist12_f64), which saves the first pass.
 *   korder_out: capacity T_cap >= T.  *n_prefix_h (HOST) = number of arcs written, or -1 when more
 *   than T_cap arcs tie at the threshold (use the full argsort then).  Synchronises the stream once.
 * The caller runs sx_kruskal on the prefix and falls back to the full order if the forest is not
 * complete within it.
 */
SX_API size_t sx_kruskal_prefix_workspace_bytes(int64_t T_cap);
SX_API int    sx_hist12_f64(const double *weight, int64_t n, uint32_t *hist12, void *stream);
SX_API int    sx_kruskal_prefix(const double *weight, int64_t n, int64_t T, int64_t T_cap,
                         const uint32_t *hist12, uint32_t *korder_out, int64_t *n_prefix_h,
                         void *ws, size_t ws_bytes, void *stream);

/* sx_order_head_sharded_h: the same head over S x D weights held as row slabs on several devices (the flow
 * scores of a row-sharded OT problem, with the row bounds of its cost slabs); one process, one host thread.
 * Every shard streams only its own weights on its own GPU; the host adds the shards' 4096-bin histograms of
 * both levels (two small round trips per shard), so every shard selects against the same threshold, and only
 * the candidates (at most T_cap arcs) are copied to devs[0], where they are sorted and ordered.
 *   devs / row_bounds: as sx_sinkhorn_ot_sharded_h (row_bounds NULL = equal partition; a device may appear more
 *     than once: its shards then run one after the other on one stream of that device, with the same results).
 *   weights[g]: DEVICE pointer on devs[g] to shard g's rows x D weights, contiguous.  Arc ids are global:
 *     row_bounds[g] * D + position in the shard; S * D >= 2^32 is SX_ERR_TOO_LARGE.
 *   hist12 (may be NULL, as may any entry): hist12[g] is shard g's level-0 histogram (sx_score_ot).
 *   mode SX_ORDER_KRUSKAL: out = uint32 ids, descending weight, ties by ascending id (sx_kruskal's input);
 *   mode SX_ORDER_QUEUE:   out = int64 ids, descending weight, ties by descending id, i.e. the head of
 *     np.argsort(w, kind="stable")[::-1] (net_manager.py:379).
 *   out: DEVICE buffer on devs[0], capacity T_cap >= T.  *n_out_h (HOST): arcs written (>= min(T, S * D)), or -1
 *     when more than T_cap arcs tie at the threshold, as sx_kruskal_prefix.
 * Blocking; allocates and frees its buffers per call (per shard 80 B x T_cap, on devs[0] ~48 B x T_cap more). */
#define SX_ORDER_KRUSKAL 0
#define SX_ORDER_QUEUE   1
SX_API int    sx_order_head_sharded_h(int ndev, const int *devs, const double *const *weights,
                               const int64_t *row_bounds, int64_t S, int64_t D, int64_t T, int64_t T_cap,
                               const uint32_t *const *hist12, int mode, void *out, int64_t *n_out_h);

/* ---- K2: spanning-tree basis identification -------------------------------------------
 * Replaces `sp.csgraph.minimum_spanning_tree(-w)` + flatnonzero, tree_BI.py:32-59.
 * Visits arcs in `korder`; keeps an arc when its end nodes are in different components
 * (lock-free union-find, path halving; chunked filter + min-rank hooking, exact because
 * the order is a strict total order); stops at N-1 arcs.  Endpoints: tail == NULL selects
 * the implicit OT graph (arc k = (k / D, S + k % D)), else tail[k], head[k].
 *   tree_out (capacity N-1): kept arc ids, ascending.  n_tree_out: their number.
 */
SX_API int    sx_kruskal_set_tuning(int first_chunk_quarters_of_N);   /* first chunk of the order = q N / 4 arcs (0: default) */
SX_API size_t sx_kruskal_workspace_bytes(int64_t N, int64_t n);
SX_API int    sx_kruskal(const uint32_t *korder, int64_t n, const int32_t *tail, const int32_t *head,
                  int64_t S, int64_t D, int64_t N, int64_t *tree_out, int64_t *n_tree_out,
                  void *ws, size_t ws_bytes, void *stream);

/* ---- K3: node potentials from the tree ------------------------------------------------
 * The reference takes duals from the LP solver (solver_caller/gurobi.py:157-159, used at
 * network_methods/algorithms.py:132); this computes them from the tree: y[root] = 0 and
 * y[plus] - y[minus] = cost for every tree arc (B^T y = c_B with B = A[:-1, tree],
 * tree_BI.py:74).  Euler tour + list ranking by pointer jumping.
 *   cost: indexed by arc id with leading dimension: cost[(k / D) * ld + k % D] when
 *   tail == NULL (dense OT cost matrix M), cost[k] otherwise.
 *   status_out (device int32): 0 or SX_ERR_NOT_SPANNING.
 *   Accuracy: exact when every cost is a multiple of one 2^-e and max|y| < 2^52 * 2^-e; otherwise
 *   |y - y_exact| <= 2 ceil(log2 H) * eps * max|y_exact| (H = 2 (N - 1)), normwise: the error of a node
 *   follows its tour position, not its root path, so relative to a small |y| it can be large.
 */
SX_API size_t sx_tree_potentials_workspace_bytes(int64_t N);
SX_API int    sx_tree_potentials(const int64_t *tree, int64_t n_tree, const int32_t *tail,
                          const int32_t *head, int64_t S, int64_t D, int64_t N,
                          const double *cost, int64_t ld, int plus_convention, int64_t root,
                          double *y_out, int32_t *status_out, void *ws, size_t ws_bytes,
                          void *stream);

/* sx_tree_flows: primal flows of the tree basis, the solution of B x = b[:-1] with B = A[:-1, tree]
 * that the reference gets from SuperLU (tree_BI.py:74-76; the dropped row is the root's).  The flow
 * on tree arc t is +/- the sum of b over the subtree below it, taken as a difference of tour-order
 * prefix sums carried in double-double.  With s the exact subtree sum and sum|b| taken over the non-root
 * nodes: |flow - s| <= ulp(s) / 2 + 2^-103 H sum|b| (H = 2 (N - 1)), hence within 1 ulp of s whenever
 * sum|b| <= 2^50 |s| / H.  A subtree whose supplies cancel exactly gets +-0.0 when the tour's prefix
 * sums are exact in double-double (supplies on one grid 2^-e spanning fewer than ~100 bits).
 *   b: N supplies (A x = b); flow_out[t] belongs to tree[t]; same workspace size and status as
 *   sx_tree_potentials.
 */
SX_API int    sx_tree_flows(const int64_t *tree, int64_t n_tree, const int32_t *tail, const int32_t *head,
                     int64_t S, int64_t D, int64_t N, const double *b, int plus_convention,
                     int64_t root, double *flow_out, int32_t *status_out, void *ws, size_t ws_bytes,
                     void *stream);

/* ---- f1 (host part): push phase of tree_basis_identify ------------------------------------
 * Replaces the loop of `push_tree_to_bfs` (tree_BI.py:81-113): for every negative tree flow (row-major
 * order, fixed before the first push) theta = first minimum of (-x[I1,J1], x[I1,J2], x[I2,J1]) is pushed
 * around the 4-cycle (I1,J1) (I2,J1) (I2,J2) (I1,J2), with J2 / I2 = np.argmax of row I1 / column J1,
 * until the flow is >= 0.  HOST buffers (the loop is sequential): tree_h (arc k = i * D + j) with its
 * primal flows flow_h (from sx_tree_flows).  Works on the sparse support (tree arcs + corners created
 * by pushes) instead of the reference's dense S x D scratch.  pos_arc_h (capacity cap): the arcs that
 * carry positive flow afterwards, i.e. vbasis == 0 (tree_BI.py:112-113), in no particular order;
 * *n_pos_h = their number (returned with SX_ERR_WORKSPACE when cap is too small: call again),
 * *push_iter_h = pushes made.  SX_ERR_PUSH_ASSERT where the reference's asserts (:93-94) would fire. */
SX_API int    sx_push_tree_h(const int64_t *tree_h, const double *flow_h, int64_t n_tree, int64_t S, int64_t D,
                      int64_t *pos_arc_h, int64_t cap, int64_t *n_pos_h, int64_t *push_iter_h);

/* ---- K4: pricing ----------------------------------------------------------------------
 * sx_price_dense_ot replaces `c - A.T @ y` + `np.all(rc >= -tol)` over the dense OT cost
 * matrix, net_manager.py:474-497:  rc_ij = fl(M_ij - fl(y_dst[j] - y_src[i])).
 *   M: rows [row0, row0 + S_loc) of the S x D cost matrix, leading dimension ld (elements);
 *   y_src: the S_loc source potentials of those rows; y_dst: the D sink potentials.
 *   Arc ids reported are global: (row0 + i) * D + j.
 *   header: counts / min (see sx_price_header).
 *   rc_out: optional full reduced-cost output (S_loc x D, ld_out), else NULL.
 *   variant: 0 = TMA-staged pipeline (needs 16 B aligned M and even ld; returns
 *   SX_ERR_UNALIGNED otherwise), 1 = vectorised direct loads, 2 = scalar loads (any
 *   alignment), -1 = choose automatically.
 * sx_price_arcs replaces net_manager.py:293-319 for an arc list:
 *   rc_k = c_k - (y[tail_k] - y[head_k]), negated where vbasis_k == -2 (+0.0 becomes -0.0).
 *   Arc ids reported are id0 + k.  16-byte aligned c / tail / head / rc_out and a 4-byte aligned
 *   vbasis take a vectorised kernel for the first E & ~3 arcs; anything else goes through the
 *   scalar one, with the same results.
 *   Its header->min_rc_key is the minimum over the reduced costs that are not NaN (+inf if all of
 *   them are, as for an empty list); a zero minimum reads +0.0, since the key does not keep the
 *   sign of zero.
 * Candidates: violators that can still be among the K most violating arcs are appended to
 *   cand_rc / cand_id (capacity cand_cap, unordered).  "Can still be" is decided from a running
 *   histogram of the appended reduced costs in `sel`, so the list stays O(K log(n / K)) long
 *   however many arcs violate; header->n_violating stays exact.  cand_cap = 0 (cand_* and sel
 *   NULL) prices for count / min only.
 * sx_price_pass_begin must be enqueued before the first sx_price_* call of a pass (it clears the
 *   header and `sel`, and records the K the pass prunes for; sel may be NULL when cand_cap = 0);
 *   several calls (row slabs, arc-list tail) may then accumulate into one header / candidate list.
 *   A pass must not price an arc twice: the selection ranks distinct (rc, id) pairs (see
 *   SX_STATUS_DUPLICATE_CANDIDATES).
 */
SX_API size_t sx_select_state_bytes(void);
SX_API int    sx_price_pass_begin(sx_price_header *header, sx_select_state *sel, int64_t K, void *stream);
SX_API int    sx_price_dense_ot(const double *M, int64_t ld, int64_t row0, int64_t S_loc, int64_t D,
                         const double *y_src, const double *y_dst, double tol,
                         sx_price_header *header, sx_select_state *sel, double *cand_rc,
                         int64_t *cand_id, int64_t cand_cap, double *rc_out, int64_t ld_out,
                         int variant, void *stream);
SX_API int    sx_price_arcs(const double *c, const int32_t *tail, const int32_t *head,
                     const int8_t *vbasis, const double *y, int64_t E, int64_t id0, double tol,
                     sx_price_header *header, sx_select_state *sel, double *cand_rc,
                     int64_t *cand_id, int64_t cand_cap, double *rc_out, void *stream);

/* Tuning knobs of sx_price_dense_ot (bench sweeps): index into the table of TMA pipeline shapes
 * {rows per box, stages, consumer warps, CTAs per SM} of variant 0 (see sx_price.cu; 0..13, default 6),
 * and the CTAs per SM of the direct-load variants (default 16).  Negative / zero values leave a knob
 * unchanged; a shape past the table is SX_ERR_INVALID.  Every accepted shape, every CTA count and every
 * option below returns the same bits: the same reduced costs, count, minimum, status and top-K
 * after selection.  They change speed only. */
SX_API int    sx_price_set_tuning(int tma_shape, int direct_ctas_per_sm);
/* TMA descriptor / cache options of variant 0: l2_promotion 0..3 = none, 64 B, 128 B, 256 B (default);
 * evict_first 1 (default) / 0 = L2 evict-first or normal policy on the loads.  Negative = unchanged,
 * l2_promotion > 3 is SX_ERR_INVALID.  Cache hints only: the results do not change. */
SX_API int    sx_price_set_tma_options(int l2_promotion, int evict_first);

/* ---- K4 fused: one launch per pricing pass -------------------------------------------------
 * sx_price_dense_ot_fused = sx_price_pass_begin + sx_price_dense_ot (variant 0) + sx_topk_select
 * (+ sx_exchange_push_ll when peer_bufs_dev != NULL) as ONE cooperative kernel: the state clear of the
 * next pass is folded into the start of this one (the pricer owns two selection states, used by
 * alternate passes), the selection runs behind two grid-wide barriers at the end of the pricing
 * pipeline, and the ranking threads store every selected arc straight into the peers' exchange
 * buffers.  Same results as the separate calls (net_manager.py:474-497 + top-k).
 *   state: sx_fused_state_bytes() bytes of device memory, 16 B aligned, initialised ONCE per pricer by
 *     sx_fused_state_init (and again after any error); K is fixed per state, 1 <= K <= SX_TOPK_MAX_K
 *     (pass cand_cap = 0 to price for count / min only).
 *   block (device, block_len >= 2 K + 6 int64): [K rc bits | K ids | n_violating, min_rc_key, n_priced,
 *     status | n_out | 0], entries past n_out are (+inf, -1).
 *   peer_bufs_dev / rank / G: as sx_exchange_push_ll (buffers of sx_exchange_ll_buffer_bytes(block_len,
 *     G) bytes).  NULL: no exchange.
 *   merged_out (device, 2 K + 5 int64, may be NULL): when given (and sx_fused_merge_fits(K, G)), the last
 *     CTAs of the same kernel also MERGE the G blocks as they land in the local buffer -- the whole
 *     multi-GPU pass is one launch per GPU: [K rc bits | K ids | n_out | total n_violating, min key,
 *     largest single n_violating, OR of the status words]; status_dev receives SX_ERR_PEER_TIMEOUT if
 *     a peer never shows up.  NULL: follow with sx_topk_merge_ll.
 *   ws: sx_topk_workspace_bytes(cand_cap, K) bytes, as sx_topk_select takes.
 * The selection is the one of sx_topk_select and finishes on any candidate list of distinct arcs.  Status bit
 * SX_STATUS_CAND_OVERFLOW asks for a larger candidate buffer and a repeat (the block is still well formed and
 * pushed, so no peer waits).  Needs 16 B aligned M and even ld (SX_ERR_UNALIGNED otherwise: use the separate
 * calls).
 */
typedef struct sx_fused_state sx_fused_state;
SX_API size_t sx_fused_state_bytes(void);
/* diagnostics: byte offset inside the state of 8 x uint64 %globaltimer stamps (ns) that CTA 0 of the last
 * pass took at: start, end of its pricing, after barrier 1, after the filter, after barrier 2, after the rank */
SX_API size_t sx_fused_state_timestamps_offset(void);
SX_API int    sx_fused_state_init(sx_fused_state *state, int64_t K, void *stream);
SX_API int    sx_fused_merge_fits(int64_t K, int G);   /* 1 when the in-kernel merge can stage G blocks of K */
SX_API int    sx_price_dense_ot_fused(const double *M, int64_t ld, int64_t row0, int64_t S_loc, int64_t D,
                               const double *y_src, const double *y_dst, double tol, sx_fused_state *state,
                               double *cand_rc, int64_t *cand_id, int64_t cand_cap, int64_t K, int64_t *block,
                               int64_t block_len, void *const *peer_bufs_dev, int rank, int G,
                               int64_t *merged_out, int32_t *status_dev, void *ws, size_t ws_bytes, void *stream);

/* ---- lower-bound copy of a cost slab: the fused pass streams 4 B per arc instead of 8 ----------
 * sx_cost_lb_build writes lb[i * ld_lb + j] = the high 32 bits of the fp64 bit pattern of M[i * ld + j],
 * rounded toward -inf (one streaming kernel).  Read back as the high half of a double with a zero low half,
 * L <= M element by element, or L is NaN:
 *   values whose low half is 0 (+-0, +-inf, and every value with at most 20 mantissa bits) are exact;
 *   other positive values truncate; other negative values step one unit away from zero (at -DBL_MAX and
 *   below: -inf); a NaN keeps its sign and exponent and gets the quiet bit (0x00080000), so it stays NaN.
 *   lb: 16 B aligned device memory, ld_lb >= D and a multiple of 4 (16 B TMA row stride); columns
 *   [D, ld_lb) are not written.  sx_cost_lb_bytes(S_loc, D) sizes a copy with ld_lb = D rounded up to 4.
 * sx_price_dense_ot_fused_lb = sx_price_dense_ot_fused (same arguments and results, bit for bit) that may
 *   stream the copy: each arc whose lower-bound reduced cost L - (v - u) is below max(running min, -tol)
 *   (or NaN) is re-read from M and priced exactly; no other arc can be a violator or a new minimum.  The
 *   copy pays off while few arcs violate, so a pass streams M itself when the previous pass on the same
 *   state had more than a fixed fraction of its arcs violating (the first pass of a state streams the
 *   copy).  lb == NULL is sx_price_dense_ot_fused.  The copy must be built from the M passed here, and M
 *   must not change while the copy is in use.
 */
SX_API size_t sx_cost_lb_bytes(int64_t S_loc, int64_t D);
SX_API int    sx_cost_lb_build(const double *M, int64_t ld, int64_t S_loc, int64_t D, uint32_t *lb, int64_t ld_lb,
                               void *stream);
SX_API int    sx_price_dense_ot_fused_lb(const double *M, int64_t ld, const uint32_t *lb, int64_t ld_lb, int64_t row0,
                                         int64_t S_loc, int64_t D, const double *y_src, const double *y_dst,
                                         double tol, sx_fused_state *state, double *cand_rc, int64_t *cand_id,
                                         int64_t cand_cap, int64_t K, int64_t *block, int64_t block_len,
                                         void *const *peer_bufs_dev, int rank, int G, int64_t *merged_out,
                                         int32_t *status_dev, void *ws, size_t ws_bytes, void *stream);

/* ---- the big-M extension priced over the base slab (replaces, for the fused pass, the extended matrix the reference
 * builds in extend_by_bigM, net_manager.py:381-400, and prices in check_optimality_condition, :474-497) ----
 * sx_price_dense_ot_fused_bigm = sx_price_dense_ot_fused_lb over rows [row0, row0 + S_loc) of an S x D base matrix
 * M, priced as that shard of the (S+1) x (D+1) extension: last column = bigM, last row = bigM, corner = `corner`.
 * A small kernel first prices the shard's border arcs (i, D) and, when row0 + S_loc == S, the artificial row (S, j),
 * j <= D, into the selection state the fused kernel then completes; the fused kernel reads the base slab as before
 * (same bytes per arc, same lower-bound copy).  Arc ids are those of the extension, i (D + 1) + j, and count,
 * minimum, NaN status and top-K are those of the physically extended matrix, bit for bit.
 *   S: base rows.  y_src: the shard's S_loc source duals.  y_dst: D + 1 sink duals (the last = the artificial
 *   sink's).  y_art: device pointer to u_S, the artificial source's dual (read only by the shard that ends at S;
 *   may be NULL on the others).  bigM / corner: the border's costs.  Everything else as sx_price_dense_ot_fused_lb.
 * Checks what sx_price_dense_ot_fused_lb checks, plus row0 + S_loc <= S and D + 1 < 2^31; on a bad argument
 * nothing is launched.
 */
SX_API int    sx_price_dense_ot_fused_bigm(const double *M, int64_t ld, const uint32_t *lb, int64_t ld_lb, int64_t row0,
                                           int64_t S_loc, int64_t S, int64_t D, const double *y_src,
                                           const double *y_dst, const double *y_art, double bigM, double corner,
                                           double tol, sx_fused_state *state, double *cand_rc, int64_t *cand_id,
                                           int64_t cand_cap, int64_t K, int64_t *block, int64_t block_len,
                                           void *const *peer_bufs_dev, int rank, int G, int64_t *merged_out,
                                           int32_t *status_dev, void *ws, size_t ws_bytes, void *stream);

/* ---- top-k most violating arcs (north_star extension; SURVEY.md section 8 row a9) -------
 * Among the candidates (rc, id) left by a pricing pass select the K smallest by (rc ascending,
 * id ascending).  sel / header are the pass's selection state and header (the candidate count
 * lives in sel).  out_rc / out_id have capacity K; out_n (device int64) = min(K, #violators).
 * Entries past out_n are filled with (+inf, -1) so fixed-size blocks can be exchanged.
 * sx_topk_select: K <= SX_TOPK_MAX_K runs the histogram filter, radix refinement of the boundary
 *   bin on (rc, id) and an all-pairs rank in one cooperative launch (no host round trip); it
 *   always finishes on distinct candidates, however many of them tie on rc.  When one (rc, id)
 *   pair at the K-th position has more copies than 8192 minus the candidates ranked before it,
 *   it raises SX_STATUS_DUPLICATE_CANDIDATES and leaves out_n = 0.  Larger K runs two stable
 *   radix argsorts (synchronises the stream once to read the candidate count).
 * sx_topk_merge merges G sorted, padded blocks (as exchanged between G ranks) into one.  Block g
 *   has its rc list at blocks_rc + g * block_stride and its ids at blocks_id + g * block_stride
 *   (strides in 8-byte elements, so the gathered buffer is consumed in place).  A block is sorted by
 *   (rc, id) as the selection writes it: its real entries, then padding (+inf, -1).  The merges
 *   (here, sx_topk_merge_ll and the in-kernel merge of sx_price_dense_ot_fused) recognise padding by
 *   id < 0, or by rc = +inf where they read only rc: a real entry is a violator, never +inf.  rc
 *   compares by its order-preserving image (-0.0 == +0.0); exact ties go to the smaller id, and ids
 *   must be distinct across blocks.  Optionally folds
 *   the G pricing headers found at headers + g * block_stride into out_summary =
 *   {total n_violating, min key, largest single n_violating, OR of the status words}.
 *   parity_ctr (device, may be NULL): when the blocks sit in a double-buffered exchange buffer
 *   (sx_exchange_blocks), the epoch counter of that buffer; the kernel then reads the half
 *   (*parity_ctr & 1), i.e. blocks_* / headers + (*parity_ctr & 1) * parity_stride, so that the
 *   launch carries no per-step argument (CUDA graphs).
 */
#define SX_TOPK_MAX_K 1024
SX_API size_t sx_topk_workspace_bytes(int64_t cand_cap, int64_t K);
SX_API int    sx_topk_select(const double *cand_rc, const int64_t *cand_id, int64_t cand_cap,
                      sx_select_state *sel, sx_price_header *header, int64_t K, double *out_rc,
                      int64_t *out_id, int64_t *out_n, void *ws, size_t ws_bytes, void *stream);
SX_API size_t sx_topk_merge_workspace_bytes(int64_t G);
SX_API int    sx_topk_merge(const double *blocks_rc, const int64_t *blocks_id, int64_t block_stride,
                     int64_t G, int64_t K, const int64_t *headers, double *out_rc, int64_t *out_id,
                     int64_t *out_n, int64_t *out_summary, const unsigned long long *parity_ctr,
                     int64_t parity_stride, void *ws, size_t ws_bytes, void *stream);

/* ---- multi-GPU exchange of the result blocks over NVLink peer memory ------------------------
 * Replaces the NCCL all-gather of the row-sharded pricing pass (no reference counterpart: the
 * reference is single process).  Every rank owns a symmetric buffer of sx_exchange_buffer_bytes()
 * bytes, zero-initialised and peer-mapped (e.g. torch symmetric memory); peer_bufs_dev is a DEVICE
 * array of the G base pointers (entry g = rank g's buffer as mapped in this process).  The buffer
 * holds [2][G][block_len] slots, [2][G] flags and, at sx_exchange_epoch_offset(), the epoch counter
 * (starts at 0; call n of every rank is epoch n).  One call stores this rank's block (block_len
 * int64, even, 16 B aligned) into slot [epoch & 1][rank] of every rank's buffer and returns (on the
 * stream) when all G blocks of this epoch have landed in the local slots [epoch & 1][0..G),
 * contiguous, block_len apart, and the local epoch counter has advanced to `epoch`.  No per-call
 * argument changes between calls, so the launch can be captured in a CUDA graph.  status_dev
 * receives SX_ERR_PEER_TIMEOUT if a peer does not show up within 10 s (never cleared by the library).
 */
SX_API size_t sx_exchange_buffer_bytes(int64_t block_len, int G);
SX_API size_t sx_exchange_epoch_offset(int64_t block_len, int G);
SX_API int    sx_exchange_blocks(const int64_t *block, int64_t block_len, void *const *peer_bufs_dev,
                          int rank, int G, int32_t *status_dev, void *stream);

/* Low-latency form of the same exchange (default of the package): sx_exchange_push_ll only STORES --
 * every 8-byte word of the block travels as one 16-byte slot {lo32, flag, hi32, flag}, flag = epoch --
 * and sx_topk_merge_ll polls the slots of its local buffer while it stages the keys of the G blocks in
 * shared memory, then merges them like sx_topk_merge.  No fence, no flag round trip, no separate wait.
 * It runs the same merge as the last CTAs of sx_price_dense_ot_fused (merged_out != NULL).
 *   Buffer: sx_exchange_ll_buffer_bytes() bytes, zeroed, peer-mapped; the epoch counters (one advanced
 *   by the pushing side, one by the merge, each once per pass) sit right after the 2 * G * block_len
 *   slots.  The merge depends on no other kernel of its GPU and is launched with programmatic stream
 *   serialisation: behind sx_price_dense_ot_fused it becomes resident while that kernel drains.  block = [K rc | K ids | 4 header words | ...], block_len >= 2 K + 4.
 *   G * K * 16 must not exceed 200 KB, else SX_ERR_TOO_LARGE (callers size against this limit; the
 *   kernel itself stages G * K * 8 bytes).
 *   out_summary (4 words, may be NULL) as in sx_topk_merge; status_dev as in sx_exchange_blocks.
 */
SX_API size_t sx_exchange_ll_buffer_bytes(int64_t block_len, int G);
SX_API int    sx_exchange_push_ll(const int64_t *block, int64_t block_len, void *const *peer_bufs_dev,
                           int rank, int G, void *stream);
SX_API int    sx_topk_merge_ll(void *ll_buf_local, int64_t block_len, int64_t G, int64_t K,
                        double *out_rc, int64_t *out_id, int64_t *out_n, int64_t *out_summary,
                        int32_t *status_dev, void *stream);

/* ---- warm start: entropic Sinkhorn point for the crossover (scripts/run_network_crossover.py:96) ----
 * The reference's OT experiments cross over `ot.sinkhorn(s, d, M, reg=10, numItermax=1000)` (POT,
 * third party, Sinkhorn-Knopp).  sx_sinkhorn_ot runs the same iteration in the log domain on the
 * device-resident cost matrix: v = b / (K^T u), u = a / (K v) from u = 1 / S, K = exp(-M / reg),
 * carried as potentials f = reg log u, g = reg log v; stops after max_iter iterations or when the
 * column-marginal error || X^T 1 - b ||_2, examined every check_every iterations, is below stop_thr
 * (<= 0: never examined).  x_out (S * D, may be NULL) receives X = exp((f_i + g_j - M_ij) / reg).
 *   f (S), g (D): device outputs.  iters_h / err_h (HOST, may be NULL): iterations run, last error.
 */
SX_API size_t sx_sinkhorn_workspace_bytes(int64_t S, int64_t D);
SX_API int    sx_sinkhorn_ot(const double *M, int64_t ld, int64_t S, int64_t D, const double *a,
                      const double *b, double reg, int64_t max_iter, double stop_thr,
                      int64_t check_every, double *f, double *g, double *x_out, int64_t *iters_h,
                      double *err_h, void *ws, size_t ws_bytes, void *stream);

/* sx_sinkhorn_ot_sharded_h: the same iteration (same order, stopping rule and check_every) over a cost matrix
 * held as row slabs on several devices, as sx_ot_pricer holds it; one process, one host thread.  Rank g runs
 * the kernels of sx_sinkhorn_ot on rows [row_bounds[g], row_bounds[g + 1]) of its slab and keeps f for them;
 * the column half-step exchanges one (max, scaled sum) log-sum-exp pair per column and rank through NVLink
 * peer stores (two 16-byte flag-in-data slots: 32 B x D from each rank into each of the G buffers per iteration),
 * and every rank merges the G pairs in rank order, so every rank computes the same g bit for bit.  The stopping
 * error is summed in a fixed order, so the iteration count does not depend on kernel timing either.  With ndev = 1 the results are those of sx_sinkhorn_ot bit for bit.
 *   devs / slabs / row_bounds / ld: as sx_ot_pricer_create (row_bounds NULL = equal partition).  A device may
 *     appear more than once: its ranks then run one after the other on one stream of that device (same
 *     results as ranks on distinct devices with the same row bounds).  Distinct devices need peer access
 *     (SX_ERR_NO_DEVICE otherwise).
 *   a_h (S), b_h (D): HOST marginals.  f_h (S), g_h (D): HOST outputs (g from rank 0).
 *   x_out (may be NULL): x_out[g] is an S_loc x D DEVICE buffer on devs[g] that receives rank g's rows of X.
 *   iters_h / err_h (HOST, may be NULL): as sx_sinkhorn_ot; the error of rank 0 decides for every rank.
 * Blocking; allocates and frees its buffers per call.  SX_ERR_PEER_TIMEOUT when a rank's pair did not arrive
 * within 10 s. */
SX_API int    sx_sinkhorn_ot_sharded_h(int ndev, const int *devs, const double *const *slabs,
                                const int64_t *row_bounds, int64_t ld, int64_t S, int64_t D, const double *a_h,
                                const double *b_h, double reg, int64_t max_iter, double stop_thr,
                                int64_t check_every, double *f_h, double *g_h, double *const *x_out,
                                int64_t *iters_h, double *err_h);

/* ---- host-buffer entry points (what a reference-side binding calls with NumPy arrays) ----
 * sx_ot_pricer: persistent pricer of one dense OT problem for `OTManager.check_optimality_condition`
 * (net_manager.py:485-497, called once per column-generation round from algorithms.py:132).  It owns every
 * buffer a pass needs (nothing is allocated per pass), one stream and one host worker thread per GPU, and
 * row-shards the cost matrix over the ndev GPUs it is given: device g prices rows [S g / ndev, S (g+1) / ndev)
 * with ONE kernel per pass (sx_price_dense_ot_fused: price + select + NVLink push + merge).  Single process,
 * plain function calls; not thread-safe (one caller at a time), like the reference's managers.
 *   slabs[g]: DEVICE pointer (on device devs[g], caller-owned, resident and unchanged for the life of the
 *     pricer) to that row range of M, row-major with leading dimension ld (even ld and 16-byte aligned slabs
 *     select the TMA / fused path; anything else is priced by the scalar-load kernels).  On the fused path
 *     the pricer builds and owns a lower-bound copy of each slab (sx_cost_lb_build, half the slab's bytes)
 *     and prices with sx_price_dense_ot_fused_lb; if that allocation fails it streams the slab itself.
 *   row_bounds (HOST, ndev + 1 entries, may be NULL): shard g holds rows [row_bounds[g], row_bounds[g + 1]);
 *     NULL = the equal partition above.  GPUs of one box stream at rates a few percent apart and a pass ends
 *     when the slowest has delivered its block, so callers may size the shards by measured rate.
 *   K: top-K size (0: count / min only).  ndev > 1 needs K <= SX_TOPK_MAX_K and peer access between the
 *     devices (SX_ERR_NO_DEVICE otherwise).
 * sx_ot_pricer_price_h: y_src_h (S source duals) and y_dst_h (D sink duals) are HOST vectors (pageable is
 *   fine: each worker copies its slice into pinned staging); returns count / min / top-K on the host and
 *   (status_h, may be NULL) the SX_STATUS_* bits that survived (SX_STATUS_NAN_RC).  Repeats the pass
 *   internally, with a larger candidate buffer, when the candidates overflowed it.
 * sx_ot_pricer_info: device / row range of shard g (base rows for a bordered pricer).  sx_ot_pricer_stats:
 *   passes, repeated passes, whether the fused kernel and the in-kernel merge are in use.
 * sx_ot_pricer_create_bigm: the same pricer over the S x D base slabs of a problem extended by big-M (reference
 *   net_manager.py:381-400: last column and last row = bigM, corner = `corner`), priced as the (S+1) x (D+1)
 *   extension with sx_price_dense_ot_fused_bigm -- the extended matrix is never built.  sx_ot_pricer_price_h then
 *   takes S + 1 source and D + 1 sink duals and returns arc ids of the extension.  Fused path only: even ld,
 *   16-byte aligned slabs (SX_ERR_UNALIGNED otherwise) and K <= SX_TOPK_MAX_K (SX_ERR_TOO_LARGE), checked before
 *   anything is allocated.
 */
typedef struct sx_ot_pricer sx_ot_pricer;
SX_API int    sx_ot_pricer_create(int ndev, const int *devs, const double *const *slabs, const int64_t *row_bounds,
                           int64_t ld, int64_t S, int64_t D, int64_t K, double tol, sx_ot_pricer **out);
SX_API int    sx_ot_pricer_create_bigm(int ndev, const int *devs, const double *const *slabs,
                                const int64_t *row_bounds, int64_t ld, int64_t S, int64_t D, double bigM,
                                double corner, int64_t K, double tol, sx_ot_pricer **out);
SX_API int    sx_ot_pricer_destroy(sx_ot_pricer *p);
SX_API int    sx_ot_pricer_info(const sx_ot_pricer *p, int g, int *dev, int64_t *row0, int64_t *S_loc);
SX_API int    sx_ot_pricer_price_h(sx_ot_pricer *p, const double *y_src_h, const double *y_dst_h,
                            unsigned long long *n_violating_h, double *min_rc_h, double *topk_rc_h,
                            int64_t *topk_id_h, int64_t *topk_n_h, unsigned long long *status_h);
SX_API int    sx_ot_pricer_stats(const sx_ot_pricer *p, unsigned long long *passes, unsigned long long *repeats,
                          int *fused, int *merge_in_kernel);

/* One-shot form: uploads y (and M if M_dev == NULL), prices on the current device, returns count / min /
 * top-k on the host.  Creates and destroys an sx_ot_pricer inside: for a single pass only -- a
 * column-generation loop holds an sx_ot_pricer.
 *   M_h: host S x D cost matrix (row-major, contiguous) or NULL when M_dev is given.
 *   M_dev: device-resident copy (leading dimension D), or NULL.
 */
SX_API int    sx_price_dense_ot_h(const double *M_h, const double *M_dev, int64_t S, int64_t D,
                           const double *y_h, double tol, int64_t K,
                           unsigned long long *n_violating_h, double *min_rc_h,
                           double *topk_rc_h, int64_t *topk_id_h, int64_t *topk_n_h);

#ifdef __cplusplus
}
#endif
#endif  /* SXCROSS_H_ */

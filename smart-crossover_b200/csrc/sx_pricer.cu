// sx_pricer.cu -- persistent dense-OT pricer behind the host-buffer entry points: one process, G GPUs.
//
// What `OTManager.check_optimality_condition` (reference net_manager.py:485-497, called from
// algorithms.py:132 once per column-generation round) needs from the device is one call: duals in (a host
// vector, as the LP solver returns it), violator count / min reduced cost / top-K out.  sx_ot_pricer keeps
// everything that call needs alive between rounds -- candidate buffers, the two selection states of the
// fused pass, exchange buffers, pinned staging, one stream and one host worker thread per GPU -- so a pass
// allocates nothing, and it row-shards the cost matrix over every GPU it was given: per GPU one host thread
// (the caller's own for device 0, a worker for each other device) uploads the duals of its rows, launches
// ONE kernel (sx_price_dense_ot_fused: price + select + NVLink push + merge) and reads the merged result
// back; the threads run concurrently, so the GPUs start within microseconds of each other and the caller
// sees a plain function call (SURVEY.md section 8e "process model").
// The cost-matrix slabs are caller-owned device memory (the managers upload M once per problem).  On the fused
// path the pricer builds one lower-bound copy per slab at create (sx_cost_lb_build: high words rounded toward
// -inf, half the slab's bytes) and the fused pass streams it while few arcs violate.
// A bordered pricer (sx_ot_pricer_create_bigm) holds the S x D base slabs and prices the (S+1) x (D+1) big-M
// extension: each pass is sx_price_dense_ot_fused_bigm, the border kernel and the fused kernel over the base slab.
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <mutex>
#include <new>
#include <string.h>
#include <thread>
#include <vector>

#include "sx_common.cuh"

namespace {

using namespace sx;

enum Cmd { kIdle = 0, kPrice = 1, kGrow = 2, kQuit = 3 };

struct DevCtx {
    int dev = 0, g = 0;
    cudaStream_t st = nullptr;
    const double *M = nullptr;
    uint32_t *lb = nullptr;                            // lower-bound copy of M (owned), or nullptr: stream M itself
    int64_t ld_lb = 0;
    int64_t row0 = 0, S_loc = 0;
    double *y_loc = nullptr;
    double *cand_rc = nullptr;
    int64_t *cand_id = nullptr;
    void *fstate = nullptr, *sel = nullptr, *topk_ws = nullptr;
    size_t topk_ws_bytes = 0;
    int64_t *block = nullptr, *merged = nullptr;
    char *ll_buf = nullptr;
    void **peer_bufs_dev = nullptr;
    double *h_y = nullptr;
    int64_t *h_out = nullptr;
    // worker thread (devices 1..G-1; device 0 is driven by the calling thread itself)
    std::thread th;
    std::mutex mu;
    std::condition_variable cv;
    std::atomic<unsigned> posted{0}, finished{0};     // sequence numbers of the last command handed over / completed
    bool sleeping = false;                            // under mu: the worker gave up spinning and waits on cv
    int cmd = kIdle, rc = SX_OK;
};

}  // namespace

struct sx_ot_pricer {
    int G = 0;
    int64_t S = 0, D = 0, ld = 0, K = 0, Kp = 1, blk = 0, cap = 0;
    double tol = 0;
    bool fusable = false, merge_in_kernel = false, dead = false;
    bool bigm = false;                                 // prices the big-M extension of the S x D base
    double bigM = 0, corner = 0;
    std::vector<DevCtx *> ctx;
    // arguments of the pass in flight (read by the workers)
    const double *y_src_h = nullptr, *y_dst_h = nullptr;
    int64_t new_cap = 0;
    unsigned long long passes = 0, repeats = 0;
};

namespace {

#define SXP(expr) do { int _r = (expr); if (_r != SX_OK) return _r; } while (0)

int alloc_candidates(sx_ot_pricer *p, DevCtx *c, int64_t cap) {
    if (c->cand_rc) cudaFree(c->cand_rc);
    if (c->cand_id) cudaFree(c->cand_id);
    if (c->topk_ws) cudaFree(c->topk_ws);
    c->cand_rc = nullptr; c->cand_id = nullptr; c->topk_ws = nullptr;
    const size_t n = (size_t)(cap > 0 ? cap : 1);
    SX_CUDA(cudaMalloc(&c->cand_rc, n * 8));
    SX_CUDA(cudaMalloc(&c->cand_id, n * 8));
    c->topk_ws_bytes = sx_topk_workspace_bytes(cap, p->Kp);
    SX_CUDA(cudaMalloc(&c->topk_ws, c->topk_ws_bytes ? c->topk_ws_bytes : 16));
    return SX_OK;
}

// One pass on one device; runs on that device's worker thread.
int run_pass(sx_ot_pricer *p, DevCtx *c) {
    const int64_t Kp = p->Kp, D = p->D, Dy = p->bigm ? D + 1 : D;
    // the duals this device needs: its own rows' source duals + every sink dual (+ u_S, the artificial source's, of
    // a bordered pricer) (pageable -> pinned) staged in chunks so that the DMA of one chunk overlaps the host copy
    // of the next (the upload of the duals is most of what a pass costs beyond the kernel: 0.5-1 MB per GPU)
    {
        const double *seg_from[3] = {p->y_src_h + c->row0, p->y_dst_h, p->y_src_h + p->S};
        const size_t seg_end[3] = {(size_t)c->S_loc, (size_t)(c->S_loc + Dy), (size_t)(c->S_loc + Dy) + (p->bigm ? 1 : 0)};
        const size_t total = seg_end[2], chunk = 16384;                      // 128 KB
        for (size_t off = 0; off < total; off += chunk) {
            const size_t len = total - off < chunk ? total - off : chunk;
            for (size_t done = 0; done < len;) {                                // [off, off + len) spans the host vectors
                const size_t pos = off + done;
                const int s = pos < seg_end[0] ? 0 : pos < seg_end[1] ? 1 : 2;
                const size_t left = seg_end[s] - pos;
                const size_t n = left < len - done ? left : len - done;
                memcpy(c->h_y + pos, seg_from[s] + (pos - (s ? seg_end[s - 1] : 0)), n * 8);
                done += n;
            }
            SX_CUDA(cudaMemcpyAsync(c->y_loc + off, c->h_y + off, len * 8, cudaMemcpyHostToDevice, c->st));
        }
    }
    const int64_t cap = p->K > 0 ? p->cap : 0;
    int32_t *xstatus = reinterpret_cast<int32_t *>(c->merged + 2 * Kp + 5);
    if (p->bigm) {
        SXP(sx_price_dense_ot_fused_bigm(c->M, p->ld, c->lb, c->ld_lb, c->row0, c->S_loc, p->S, D, c->y_loc,
                                         c->y_loc + c->S_loc, c->y_loc + c->S_loc + Dy, p->bigM, p->corner, p->tol,
                                         (sx_fused_state *)c->fstate, c->cand_rc, c->cand_id, cap, Kp, c->block, p->blk,
                                         p->G > 1 ? c->peer_bufs_dev : nullptr, c->g, p->G,
                                         (p->G > 1 && p->merge_in_kernel) ? c->merged : nullptr, xstatus, c->topk_ws,
                                         c->topk_ws_bytes, c->st));
    } else if (p->fusable) {
        SXP(sx_price_dense_ot_fused_lb(c->M, p->ld, c->lb, c->ld_lb, c->row0, c->S_loc, D, c->y_loc,
                                       c->y_loc + c->S_loc, p->tol, (sx_fused_state *)c->fstate, c->cand_rc,
                                       c->cand_id, cap, Kp, c->block, p->blk, p->G > 1 ? c->peer_bufs_dev : nullptr,
                                       c->g, p->G, (p->G > 1 && p->merge_in_kernel) ? c->merged : nullptr, xstatus,
                                       c->topk_ws, c->topk_ws_bytes, c->st));
    } else {
        sx_price_header *hdr = reinterpret_cast<sx_price_header *>(c->block + 2 * Kp);
        SXP(sx_price_pass_begin(hdr, (sx_select_state *)c->sel, p->K, c->st));
        SXP(sx_price_dense_ot(c->M, p->ld, c->row0, c->S_loc, D, c->y_loc, c->y_loc + c->S_loc, p->tol, hdr,
                              (sx_select_state *)c->sel, c->cand_rc, c->cand_id, cap, nullptr, 0, -1, c->st));
        if (p->K > 0) {
            SXP(sx_topk_select(c->cand_rc, c->cand_id, cap, (sx_select_state *)c->sel, hdr, p->K, (double *)c->block,
                               c->block + Kp, c->block + 2 * Kp + 4, c->topk_ws, c->topk_ws_bytes, c->st));
        }
        if (p->G > 1) SXP(sx_exchange_push_ll(c->block, p->blk, c->peer_bufs_dev, c->g, p->G, c->st));
    }
    if (p->G > 1 && !(p->fusable && p->merge_in_kernel))
        SXP(sx_topk_merge_ll(c->ll_buf, p->blk, p->G, Kp, (double *)c->merged, c->merged + Kp, c->merged + 2 * Kp,
                             c->merged + 2 * Kp + 1, xstatus, c->st));
    SX_CUDA(cudaMemcpyAsync(c->h_out, p->G > 1 ? c->merged : c->block, (size_t)p->blk * 8, cudaMemcpyDeviceToHost, c->st));
    SX_CUDA(cudaStreamSynchronize(c->st));
    return SX_OK;
}

int do_cmd(sx_ot_pricer *p, DevCtx *c, int cmd) {
    if (cmd == kPrice) return run_pass(p, c);
    if (cmd == kGrow) return alloc_candidates(p, c, p->new_cap);
    return SX_OK;
}

// A worker spins for its next command for a short while after finishing one -- passes of a benchmark loop or
// of a fast column-generation round follow each other within microseconds, and a futex wake-up costs 20-50 us,
// a third of a pass over a 0.4 GB slab -- and then sleeps on the condition variable.
constexpr long long kSpinNs = 200 * 1000;

void worker(sx_ot_pricer *p, DevCtx *c) {
    cudaSetDevice(c->dev);
    unsigned last = 0;
    for (;;) {
        const unsigned want = last + 1;
        const auto t0 = std::chrono::steady_clock::now();
        while (c->posted.load(std::memory_order_acquire) != want) {
            if (std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0).count() > kSpinNs) {
                std::unique_lock<std::mutex> lk(c->mu);
                c->sleeping = true;
                c->cv.wait(lk, [&] { return c->posted.load(std::memory_order_acquire) == want; });
                c->sleeping = false;
                break;
            }
#if defined(__x86_64__)
            __builtin_ia32_pause();
#endif
        }
        last = want;
        const int cmd = c->cmd;
        c->rc = do_cmd(p, c, cmd);
        c->finished.store(want, std::memory_order_release);
        if (cmd == kQuit) return;
    }
}

void post(DevCtx *c, int cmd) {
    c->cmd = cmd;
    c->posted.store(c->posted.load(std::memory_order_relaxed) + 1, std::memory_order_release);
    std::lock_guard<std::mutex> lk(c->mu);
    if (c->sleeping) c->cv.notify_all();
}

// Hand `cmd` to every worker, run device 0's share on the calling thread, wait for the workers (they finish
// within microseconds of device 0: every GPU runs the same pass); the first error code wins.
int run_all(sx_ot_pricer *p, int cmd) {
    for (size_t g = 1; g < p->ctx.size(); ++g) post(p->ctx[g], cmd);
    int prev = 0;
    cudaGetDevice(&prev);
    cudaSetDevice(p->ctx[0]->dev);
    int rc = do_cmd(p, p->ctx[0], cmd);
    cudaSetDevice(prev);
    for (size_t g = 1; g < p->ctx.size(); ++g) {
        DevCtx *c = p->ctx[g];
        const unsigned want = c->posted.load(std::memory_order_relaxed);
        while (c->finished.load(std::memory_order_acquire) != want) {
#if defined(__x86_64__)
            __builtin_ia32_pause();
#endif
        }
        if (rc == SX_OK && c->rc != SX_OK) rc = c->rc;
    }
    return rc;
}

void free_ctx(DevCtx *c) {
    cudaSetDevice(c->dev);
    if (c->st) cudaStreamSynchronize(c->st);
    void *dev_ptrs[] = {c->y_loc, c->cand_rc, c->cand_id, c->fstate, c->sel, c->topk_ws, c->block, c->merged, c->ll_buf,
                        c->peer_bufs_dev, c->lb};
    for (void *q : dev_ptrs) if (q) cudaFree(q);
    if (c->h_y) cudaFreeHost(c->h_y);
    if (c->h_out) cudaFreeHost(c->h_out);
    if (c->st) cudaStreamDestroy(c->st);
    delete c;
}

}  // namespace

extern "C" int sx_ot_pricer_destroy(sx_ot_pricer *p) {
    if (!p) return SX_OK;
    int prev = 0;
    cudaGetDevice(&prev);
    for (DevCtx *c : p->ctx) {
        if (c->th.joinable()) {
            post(c, kQuit);
            c->th.join();
        }
    }
    for (DevCtx *c : p->ctx) free_ctx(c);
    cudaSetDevice(prev);
    delete p;
    return SX_OK;
}

namespace {

struct Border { double bigM, corner; };

// want_lb: build the lower-bound copies (a pricer that prices once, sx_price_dense_ot_h, would only pay for them).
// bm: price the big-M extension of the S x D slabs (fused path only).
int ot_pricer_create(int ndev, const int *devs, const double *const *slabs, const int64_t *row_bounds, int64_t ld,
                     int64_t S, int64_t D, int64_t K, double tol, bool want_lb, const Border *bm, sx_ot_pricer **out) {
    if (!out) return SX_ERR_INVALID;
    *out = nullptr;
    if (ndev < 1 || ndev > 64 || !devs || !slabs || S < 1 || D < 1 || ld < D || K < 0) return SX_ERR_INVALID;
    if (ndev > S) return SX_ERR_INVALID;                      // every device needs at least one row
    if (row_bounds) {
        if (row_bounds[0] != 0 || row_bounds[ndev] != S) return SX_ERR_INVALID;
        for (int g = 0; g < ndev; ++g) if (row_bounds[g + 1] <= row_bounds[g]) return SX_ERR_INVALID;
    }
    const int64_t Kp = K > 0 ? K : 1;
    if (bm) {                                                 // the bordered form runs on the fused path only
        for (int g = 0; g < ndev; ++g) if (!slabs[g]) return SX_ERR_INVALID;
        if (Kp > SX_TOPK_MAX_K || D + 1 >= (1ll << 31)) return SX_ERR_TOO_LARGE;
        if (ld % 2 != 0) return SX_ERR_UNALIGNED;
        for (int g = 0; g < ndev; ++g) if (((uintptr_t)slabs[g] & 15) != 0) return SX_ERR_UNALIGNED;
    }
    if (ndev > 1 && (K > SX_TOPK_MAX_K || (size_t)16 * ndev * Kp > 200 * 1024)) return SX_ERR_TOO_LARGE;
    int prev = 0;
    SX_CUDA(cudaGetDevice(&prev));
    sx_ot_pricer *p = new (std::nothrow) sx_ot_pricer();
    if (!p) return SX_ERR_INVALID;
    p->G = ndev; p->S = S; p->D = D; p->ld = ld; p->K = K; p->Kp = Kp; p->tol = tol;
    p->blk = 2 * Kp + 6;
    p->cap = K > 0 ? (64 * K > (1ll << 20) ? 64 * K : (1ll << 20)) : 0;
    p->fusable = (ld % 2 == 0) && Kp <= SX_TOPK_MAX_K;
    p->bigm = bm != nullptr;
    if (bm) { p->bigM = bm->bigM; p->corner = bm->corner; }
    const int64_t n_y = D + (bm ? 2 : 0);                     // staged duals beyond the shard's sources
    p->merge_in_kernel = ndev > 1 && sx_fused_merge_fits(Kp, ndev);
    int rc = SX_OK;
    auto fail = [&](int code) { cudaSetDevice(prev); sx_ot_pricer_destroy(p); return code; };
    for (int g = 0; g < ndev; ++g) {
        DevCtx *c = new (std::nothrow) DevCtx();
        if (!c) return fail(SX_ERR_INVALID);
        p->ctx.push_back(c);
        c->dev = devs[g]; c->g = g;
        c->row0 = row_bounds ? row_bounds[g] : S * g / ndev;
        c->S_loc = (row_bounds ? row_bounds[g + 1] : S * (g + 1) / ndev) - c->row0;
        c->M = slabs[g];
        if (!c->M) return fail(SX_ERR_INVALID);
        if (((uintptr_t)c->M & 15) != 0) p->fusable = false;
        if (cudaSetDevice(c->dev) != cudaSuccess) return fail(SX_ERR_NO_DEVICE);
        if (ndev > 1) {
            // one GPU per shard: the ranks of a pass wait for each other inside one kernel
            for (int h = 0; h < ndev; ++h) if (h != g && devs[h] == c->dev) return fail(SX_ERR_NO_DEVICE);
            if ((rc = enable_peer_access(c->dev, ndev, devs)) != SX_OK) return fail(rc);
        }
#define SXA(call) do { cudaError_t _e = (call); if (_e != cudaSuccess) return fail(cuda_fail(_e)); } while (0)
        SXA(cudaStreamCreateWithFlags(&c->st, cudaStreamNonBlocking));
        SXA(cudaMalloc(&c->y_loc, (size_t)(c->S_loc + n_y) * 8));
        SXA(cudaMalloc(&c->block, (size_t)p->blk * 8));
        SXA(cudaMalloc(&c->merged, (size_t)p->blk * 8));
        SXA(cudaMemsetAsync(c->block, 0, (size_t)p->blk * 8, c->st));
        SXA(cudaMemsetAsync(c->merged, 0, (size_t)p->blk * 8, c->st));
        SXA(cudaMalloc(&c->sel, sx_select_state_bytes()));
        SXA(cudaMemsetAsync(c->sel, 0, sx_select_state_bytes(), c->st));
        if ((rc = alloc_candidates(p, c, p->cap)) != SX_OK) return fail(rc);
        if (p->fusable) {
            SXA(cudaMalloc(&c->fstate, sx_fused_state_bytes()));
            if ((rc = sx_fused_state_init((sx_fused_state *)c->fstate, Kp, c->st)) != SX_OK) return fail(rc);
        }
        if (p->fusable && want_lb) {
            c->ld_lb = (D + 3) & ~(int64_t)3;
            if (cudaMalloc((void **)&c->lb, sx_cost_lb_bytes(c->S_loc, D)) != cudaSuccess) {
                cudaGetLastError();                                    // no room for the copy: stream M itself
                c->lb = nullptr;
            } else if ((rc = sx_cost_lb_build(c->M, ld, c->S_loc, D, c->lb, c->ld_lb, c->st)) != SX_OK) {
                return fail(rc);
            }
        }
        if (ndev > 1) {
            const size_t nb = sx_exchange_ll_buffer_bytes(p->blk, ndev);
            SXA(cudaMalloc((void **)&c->ll_buf, nb));
            SXA(cudaMemsetAsync(c->ll_buf, 0, nb, c->st));
            SXA(cudaMalloc((void **)&c->peer_bufs_dev, sizeof(void *) * ndev));
        }
        SXA(cudaHostAlloc((void **)&c->h_y, (size_t)(c->S_loc + n_y) * 8, cudaHostAllocDefault));
        SXA(cudaHostAlloc((void **)&c->h_out, (size_t)p->blk * 8, cudaHostAllocDefault));
        SXA(cudaStreamSynchronize(c->st));
    }
    if (ndev > 1) {                                             // every device learns every exchange buffer
        std::vector<void *> bufs(ndev);
        for (int g = 0; g < ndev; ++g) bufs[g] = p->ctx[g]->ll_buf;
        for (DevCtx *c : p->ctx) {
            if (cudaSetDevice(c->dev) != cudaSuccess) return fail(SX_ERR_NO_DEVICE);
            SXA(cudaMemcpy(c->peer_bufs_dev, bufs.data(), sizeof(void *) * ndev, cudaMemcpyHostToDevice));
        }
    }
#undef SXA
    for (size_t g = 1; g < p->ctx.size(); ++g) p->ctx[g]->th = std::thread(worker, p, p->ctx[g]);
    cudaSetDevice(prev);
    *out = p;
    return SX_OK;
}

}  // namespace

extern "C" int sx_ot_pricer_create(int ndev, const int *devs, const double *const *slabs, const int64_t *row_bounds,
                                   int64_t ld, int64_t S, int64_t D, int64_t K, double tol, sx_ot_pricer **out) {
    return ot_pricer_create(ndev, devs, slabs, row_bounds, ld, S, D, K, tol, /*want_lb=*/true, nullptr, out);
}

extern "C" int sx_ot_pricer_create_bigm(int ndev, const int *devs, const double *const *slabs,
                                        const int64_t *row_bounds, int64_t ld, int64_t S, int64_t D, double bigM,
                                        double corner, int64_t K, double tol, sx_ot_pricer **out) {
    const Border bm{bigM, corner};
    return ot_pricer_create(ndev, devs, slabs, row_bounds, ld, S, D, K, tol, /*want_lb=*/true, &bm, out);
}

extern "C" int sx_ot_pricer_info(const sx_ot_pricer *p, int g, int *dev, int64_t *row0, int64_t *S_loc) {
    if (!p || g < 0 || g >= p->G) return SX_ERR_INVALID;
    if (dev) *dev = p->ctx[g]->dev;
    if (row0) *row0 = p->ctx[g]->row0;
    if (S_loc) *S_loc = p->ctx[g]->S_loc;
    return SX_OK;
}

extern "C" int sx_ot_pricer_price_h(sx_ot_pricer *p, const double *y_src_h, const double *y_dst_h,
                                    unsigned long long *n_violating_h, double *min_rc_h, double *topk_rc_h,
                                    int64_t *topk_id_h, int64_t *topk_n_h, unsigned long long *status_h) {
    if (!p || !y_src_h || !y_dst_h || !n_violating_h || !min_rc_h) return SX_ERR_INVALID;
    if (p->K > 0 && (!topk_rc_h || !topk_id_h || !topk_n_h)) return SX_ERR_INVALID;
    if (p->dead) return SX_ERR_PEER_TIMEOUT;
    const int64_t Kp = p->Kp;
    p->y_src_h = y_src_h; p->y_dst_h = y_dst_h;
    ++p->passes;
    unsigned long long status = 0, count = 0, cmax = 0;
    long long min_key = 0;
    int64_t n_out = 0;
    const int64_t kMaxCap = 1ll << 28;
    for (;;) {
        SXP(run_all(p, kPrice));
        const int64_t *h = p->ctx[0]->h_out;
        if (p->G > 1) {
            const int xs = (int)(h[2 * Kp + 5] & 0xffffffffll);
            if (xs != 0) { p->dead = true; return xs; }            // epochs may be out of step now
            n_out = h[2 * Kp]; count = (unsigned long long)h[2 * Kp + 1]; min_key = h[2 * Kp + 2];
            cmax = (unsigned long long)h[2 * Kp + 3]; status = (unsigned long long)h[2 * Kp + 4];
        } else {
            count = (unsigned long long)h[2 * Kp]; min_key = h[2 * Kp + 1]; status = (unsigned long long)h[2 * Kp + 3];
            n_out = h[2 * Kp + 4]; cmax = count;
        }
        if (p->K == 0 || (status & SX_STATUS_CAND_OVERFLOW) == 0) break;
        // the candidate buffer overflowed on some device: every device grows it and prices again
        ++p->repeats;
        if (p->cap >= kMaxCap) return SX_ERR_TOO_LARGE;
        int64_t cap = 4 * p->cap > 1024 ? 4 * p->cap : 1024;
        if (cap > kMaxCap) cap = kMaxCap;
        if (cmax && (int64_t)cmax < cap) cap = (int64_t)cmax > 1024 ? (int64_t)cmax : 1024;
        p->new_cap = cap;
        SXP(run_all(p, kGrow));
        p->cap = cap;
    }
    *n_violating_h = count;
    *min_rc_h = min_key_to_f64(min_key);
    if (status_h) *status_h = status;
    if (p->K > 0) {
        const int64_t *h = p->ctx[0]->h_out;
        if (n_out < 0) n_out = 0;
        if (n_out > p->K) n_out = p->K;
        memcpy(topk_rc_h, h, (size_t)n_out * 8);
        memcpy(topk_id_h, h + Kp, (size_t)n_out * 8);
        *topk_n_h = n_out;
    }
    return SX_OK;
}

extern "C" int sx_ot_pricer_stats(const sx_ot_pricer *p, unsigned long long *passes, unsigned long long *repeats,
                                  int *fused, int *merge_in_kernel) {
    if (!p) return SX_ERR_INVALID;
    if (passes) *passes = p->passes;
    if (repeats) *repeats = p->repeats;
    if (fused) *fused = p->fusable ? 1 : 0;
    if (merge_in_kernel) *merge_in_kernel = p->merge_in_kernel ? 1 : 0;
    return SX_OK;
}

// One-shot form of the same call (uploads M when M_dev == NULL, creates and destroys a pricer): kept for
// callers that price once; a column-generation loop should hold an sx_ot_pricer instead.
extern "C" int sx_price_dense_ot_h(const double *M_h, const double *M_dev, int64_t S, int64_t D,
                                   const double *y_h, double tol, int64_t K,
                                   unsigned long long *n_violating_h, double *min_rc_h,
                                   double *topk_rc_h, int64_t *topk_id_h, int64_t *topk_n_h) {
    if ((!M_h && !M_dev) || !y_h || S <= 0 || D <= 0 || K < 0 || !n_violating_h || !min_rc_h) return SX_ERR_INVALID;
    if (K > 0 && (!topk_rc_h || !topk_id_h || !topk_n_h)) return SX_ERR_INVALID;
    int dev = 0;
    SX_CUDA(cudaGetDevice(&dev));
    double *M_up = nullptr;
    int64_t ld = D;
    if (!M_dev) {
        ld = D + (D & 1);                                        // even leading dimension: TMA path
        SX_CUDA(cudaMalloc((void **)&M_up, (size_t)S * ld * 8));
        cudaError_t e = cudaMemcpy2D(M_up, (size_t)ld * 8, M_h, (size_t)D * 8, (size_t)D * 8, (size_t)S,
                                     cudaMemcpyHostToDevice);
        if (e != cudaSuccess) { cudaFree(M_up); return cuda_fail(e); }
        M_dev = M_up;
    }
    sx_ot_pricer *p = nullptr;
    const double *slabs[1] = {M_dev};
    int rc = ot_pricer_create(1, &dev, slabs, nullptr, ld, S, D, K, tol, /*want_lb=*/false, nullptr, &p);
    if (rc == SX_OK) {
        rc = sx_ot_pricer_price_h(p, y_h, y_h + S, n_violating_h, min_rc_h, topk_rc_h, topk_id_h, topk_n_h, nullptr);
        sx_ot_pricer_destroy(p);
    }
    if (M_up) cudaFree(M_up);
    return rc;
}

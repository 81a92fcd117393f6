"""Row-sharded dense OT pricing across GPUs (one process per GPU, `torch.distributed` / NCCL).

BASELINE.json north_star: "Dense OT pricing is row-sharded across the 8 B200s, with the
local top-k candidates merged by an NCCL allgather over NVLink, while the tree build and
potentials stay on one GPU."  Rank g owns rows [row0, row0 + S_loc) of the S x D cost matrix
as one contiguous slab in its HBM; a pricing pass is

    y (S + D fp64, <= 1 MB) on every rank
      -> sx_price_dense_ot over the slab   (count, min, violator compaction)
      -> sx_topk_select                    (local K best, padded block)
      -> exchange of one packed block per rank: K rc + K ids + header = 16 K + 48 B
         (NVLink peer stores, sx_exchange_blocks; or an NCCL all-gather)
      -> sx_topk_merge over the G blocks   (all-pairs rank; result independent of G)

With world size 1 the collective and the merge are skipped.  The reference has no
counterpart (single process, `net_manager.py:485-497` prices every arc on one core).
"""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist

from .. import device as dev
from .. import _native
from .._native import check, lib


def row_partition(S: int, world: int, rank: int):
    """Contiguous, balanced row range of `rank`: rows [S*rank/world, S*(rank+1)/world)."""
    lo = S * rank // world
    hi = S * (rank + 1) // world
    return lo, hi - lo


def block_views(gathered: torch.Tensor, K: int):
    """Views into the gathered (G, 2K+6) int64 buffer: (G, K) rc, (G, K) ids, (G, 4) headers.
    Each rank's row is its `Pricer.block` = [K rc bits | K ids | n_violating, min key, n_priced, status | n_out, -]."""
    return gathered[:, :K].view(torch.float64), gathered[:, K:2 * K], gathered[:, 2 * K:2 * K + 4]


class ShardedDensePricer:
    """Pricing of one row slab per rank + global top-K.  `M_loc` is this rank's slab (S_loc x D,
    row-major, device resident for the life of the problem, like the reference keeps `ot.M`)."""

    def __init__(self, M_loc: torch.Tensor, S: int, row0: int, K: int, tol: float = dev.TOL_RC,
                 group=None, variant: int = -1, exchange: str = "ll", use_graph: bool = True, fused: bool | None = None,
                 fused_merge: bool = True):
        self.M = M_loc
        self.S, self.D = int(S), int(M_loc.shape[1])
        self.S_loc, self.row0 = int(M_loc.shape[0]), int(row0)
        self.K, self.tol, self.variant = int(K), float(tol), variant
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        self.fused = bool(dev.FUSED_DEFAULT if fused is None else fused) and variant in (-1, 0) and dev.Pricer.fusable(M_loc, M_loc.stride(0)) \
            and max(self.K, 1) <= _native.SX_TOPK_MAX_K and self.S_loc > 0
        self.pricer = dev.Pricer(M_loc.device, self.K, fused=self.fused)
        self._merge_launches = 0
        self._dead = False
        self.use_graph = bool(use_graph)
        self._graph, self._capture_tried, self._graph_launches, self._replayed_launches = None, False, 0, 0
        self._capture_overcount = 0
        self.y_loc = torch.empty(self.S_loc + self.D, dtype=torch.float64, device=M_loc.device)
        # pinned staging of the full dual vector; `y_pinned` hands it to callers that can write their duals
        # straight into it (the solver's output buffer) and so skip one host-side copy per pass
        self.h_y = torch.zeros(self.S + self.D, dtype=torch.float64).pin_memory()
        self._h_y_np = self.h_y.numpy()
        Kp = max(self.K, 1)
        self.blk = 2 * Kp + dev.Pricer.BLOCK_TAIL
        self.gathered = torch.empty(self.world, self.blk, dtype=torch.int64, device=M_loc.device)
        # merged result: [K rc | K ids | n_out | total count, min key, largest per-rank count, status | exchange status]
        self.h_out = torch.empty(2 * Kp + 6, dtype=torch.int64).pin_memory()
        self.d_out = torch.zeros(2 * Kp + 6, dtype=torch.int64, device=M_loc.device)
        self._xstatus = self.d_out[2 * Kp + 5:2 * Kp + 6].view(torch.int32)[:1]   # written by the exchange / merge kernels
        self._merge_ws = dev._ws(lib.sx_topk_merge_workspace_bytes(self.world), M_loc.device)
        self._m_rc = self.d_out[:Kp].view(torch.float64)
        self._m_id = self.d_out[Kp:2 * Kp]
        self._m_n = self.d_out[2 * Kp:2 * Kp + 1]
        self._m_sum = self.d_out[2 * Kp + 1:2 * Kp + 5]
        # exchange of the result blocks over NVLink peer memory (torch symmetric memory):
        #   "ll"   flag-in-data stores, polled by the merge kernel itself (sx_exchange_push_ll + sx_topk_merge_ll)
        #   "p2p"  stores + release flag + wait kernel (sx_exchange_blocks), then sx_topk_merge
        #   "nccl" all_gather_into_tensor, then sx_topk_merge
        self.exchange = exchange if self.world > 1 else "none"
        if self.exchange == "ll" and 16 * self.world * Kp > 200 * 1024:
            self.exchange = "p2p"                       # blocks do not fit the merge kernel's shared memory
        if self.exchange in ("ll", "p2p"):
            err = None
            try:
                self._setup_p2p(Kp)
            except Exception as e:                      # no peer access on this box
                err = e
            # every rank must use the same exchange: one rank falling back alone would leave the others
            # spinning on its slots (all_reduce MIN of the success flags)
            ok = torch.tensor([0 if err is not None else 1], dtype=torch.int32, device=M_loc.device)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)   # also the barrier after the zero-fill
            if int(ok.item()) == 0:
                import warnings
                warnings.warn("NVLink peer exchange unavailable on at least one rank"
                              + (f" ({type(err).__name__}: {err})" if err is not None else "")
                              + "; every rank uses the NCCL all-gather")
                self.exchange = "nccl"

        # fused pass + "ll" exchange: the merge of the G blocks runs inside the same kernel when they fit
        self.fused_merge = bool(fused_merge) and self.fused and self.exchange == "ll" \
            and bool(lib.sx_fused_merge_fits(Kp, self.world))

    def _setup_p2p(self, Kp: int):
        import torch.distributed._symmetric_memory as symm
        blk = self.blk
        if self.exchange == "ll":
            n64 = lib.sx_exchange_ll_buffer_bytes(blk, self.world) // 8
        else:
            n64 = lib.sx_exchange_buffer_bytes(blk, self.world) // 8
        self._symm = symm.empty(n64, dtype=torch.int64, device=self.M.device)
        self._symm.zero_()
        torch.cuda.synchronize()
        self._hdl = symm.rendezvous(self._symm, group=self.group if self.group is not None else dist.group.WORLD)
        self._rank = dist.get_rank(self.group)
        if self.exchange == "p2p":
            off = lib.sx_exchange_epoch_offset(blk, self.world) // 8
            self._epoch_ctr = self._symm[off:off + 1]

    @property
    def stage_names(self):
        """Names of the intervals between the `stage_events` of `enqueue`."""
        if self.fused:
            return ["fused begin+pricing+selection" + ("+push" if self.exchange == "ll" else "")
                    + ("+merge" if self.fused_merge else ""), "selection", "exchange", "merge"]
        return ["begin+pricing", "selection", "exchange", "merge"]

    @property
    def pricing_kernel_name(self):
        if self.fused:
            return "price_fused_kernel"
        return "price_dense_tma_kernel" if self.variant in (-1, 0) else "price_dense_direct_kernel"

    @property
    def launches(self):
        """Kernels of libsxcross enqueued by this object."""
        return self.pricer.launches + self._merge_launches + self._replayed_launches - self._capture_overcount

    # -- device-only step: everything stays on the GPU(s) --------------------------------------
    def enqueue(self, y_dev: torch.Tensor, kernel_events=None, stage_events=None, y_parts=None):
        """Enqueue one pricing pass; returns device tensors
        (rc[K], id[K], n_out, count, min key, largest per-rank count, status).  A status with
        SX_STATUS_CAND_OVERFLOW means the pass must be repeated with larger candidate buffers (`price`
        does that).  `kernel_events` =
        (start, end) CUDA events recorded around the pricing kernel launch (bench.py's roofline
        measurement); `stage_events` = 5 events recorded at pass start, after pricing, after the
        selection, after the exchange and after the merge (the last two only when world > 1).
        `y_parts` = (source duals of this rank's rows, sink duals) replaces the slices of `y_dev`."""
        p = self.pricer
        y_src, y_dst = y_parts if y_parts is not None else (y_dev[self.row0:self.row0 + self.S_loc],
                                                              y_dev[self.S:self.S + self.D])
        mark = (lambda i: stage_events[i].record()) if stage_events is not None else (lambda i: None)
        mark(0)
        if self.fused:
            # ONE launch: state clear of the next pass, pricing, selection and (exchange "ll") the push of the
            # selected arcs into every peer's buffer
            if kernel_events is not None:
                kernel_events[0].record()
            if self.exchange == "ll":
                p.price_dense_fused(self.M, self.M.stride(0), self.row0, self.S_loc, self.D, y_src, y_dst, self.tol,
                                    self._hdl.buffer_ptrs_dev, self._rank, self.world,
                                    merged=self.d_out if self.fused_merge else None,
                                    xstatus=self._xstatus if self.fused_merge else None)
            else:
                p.price_dense_fused(self.M, self.M.stride(0), self.row0, self.S_loc, self.D, y_src, y_dst, self.tol)
            if kernel_events is not None:
                kernel_events[1].record()
            mark(1)
        else:
            p.reset()
            if kernel_events is not None:
                kernel_events[0].record()
            p.price_dense(self.M, self.M.stride(0), self.row0, self.S_loc, self.D, y_src, y_dst,
                          self.tol, None, self.variant)
            if kernel_events is not None:
                kernel_events[1].record()
            mark(1)
            p.select()
        mark(2)
        Kp = max(self.K, 1)
        if self.world == 1:
            return p.out_rc, p.out_id, p.out_n[0], p.header[0], p.header[1], p.header[0], p.header[3]
        # one exchange: every rank's block (top-K + header) lands in `gathered`, consumed in place
        if self.exchange == "ll":
            if self.fused_merge:                           # the merge ran inside the pricing kernel too
                mark(3)
                mark(4)
                return (self._m_rc, self._m_id, self._m_n[0], self._m_sum[0], self._m_sum[1], self._m_sum[2],
                        self._m_sum[3])
            if not self.fused:
                check(lib.sx_exchange_push_ll(dev._ptr(p.block), self.blk, self._hdl.buffer_ptrs_dev, self._rank,
                                              self.world, dev._stream()), "sx_exchange_push_ll")
                self._merge_launches += 1
            mark(3)
            check(lib.sx_topk_merge_ll(dev._ptr(self._symm), self.blk, self.world, Kp, dev._ptr(self._m_rc),
                                       dev._ptr(self._m_id), dev._ptr(self._m_n), dev._ptr(self._m_sum),
                                       dev._ptr(self._xstatus), dev._stream()), "sx_topk_merge_ll")
            self._merge_launches += 1
            mark(4)
            return (self._m_rc, self._m_id, self._m_n[0], self._m_sum[0], self._m_sum[1], self._m_sum[2],
                    self._m_sum[3])
        if self.exchange == "p2p":
            check(lib.sx_exchange_blocks(dev._ptr(p.block), self.blk, self._hdl.buffer_ptrs_dev, self._rank,
                                         self.world, dev._ptr(self._xstatus), dev._stream()), "sx_exchange_blocks")
            self._merge_launches += 1
            # both halves of the double buffer are passed; the merge kernel picks (epoch & 1) on the device
            gathered = self._symm[:self.world * self.blk].view(self.world, self.blk)
            parity_ctr, parity_stride = dev._ptr(self._epoch_ctr), self.world * self.blk
        else:
            dist.all_gather_into_tensor(self.gathered.view(-1), p.block, group=self.group)
            gathered = self.gathered
            parity_ctr, parity_stride = None, 0
        mark(3)
        rc, ids, hdr = block_views(gathered, Kp)
        check(lib.sx_topk_merge(dev._ptr(rc), dev._ptr(ids), gathered.stride(0), self.world, Kp, dev._ptr(hdr),
                                dev._ptr(self._m_rc), dev._ptr(self._m_id), dev._ptr(self._m_n), dev._ptr(self._m_sum),
                                parity_ctr, parity_stride,
                                dev._ptr(self._merge_ws), self._merge_ws.numel(), dev._stream()), "sx_topk_merge")
        self._merge_launches += 1
        mark(4)
        return self._m_rc, self._m_id, self._m_n[0], self._m_sum[0], self._m_sum[1], self._m_sum[2], self._m_sum[3]

    # -- host-facing call: duals in, (count, min, top-K) out --------------------------------------
    def _step(self):
        """H2D of the duals this rank needs (its rows + every sink), one pass, D2H of the result."""
        r0 = self.row0                                             # y_loc = [this rank's S_loc source duals | D sink duals]
        self.y_loc[:self.S_loc].copy_(self.h_y[r0:r0 + self.S_loc], non_blocking=True)
        self.y_loc[self.S_loc:].copy_(self.h_y[self.S:], non_blocking=True)
        self.enqueue(None, y_parts=(self.y_loc[:self.S_loc], self.y_loc[self.S_loc:]))
        if self.world == 1:
            self.pricer.h_block.copy_(self.pricer.block, non_blocking=True)
        else:
            self.h_out.copy_(self.d_out, non_blocking=True)        # result, summary and exchange status in one copy

    def _capture(self):
        """Record one step (copies + kernels) in a CUDA graph: one launch call per pass instead of ~8.
        NCCL exchange stays eager."""
        self._graph = None
        if not self.use_graph or self.exchange == "nccl":
            return
        cur = torch.cuda.current_stream()
        side = torch.cuda.Stream()
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            self._step()                                   # warm-up outside the capture (lazy module loads)
        cur.wait_stream(side)
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier(group=self.group)                 # every rank did the same number of exchanges
        launches = self.launches
        g = torch.cuda.CUDAGraph()
        try:
            with torch.cuda.graph(g):
                self._step()
        except Exception as e:                             # capture refused (driver / allocator state): stay eager
            import warnings
            warnings.warn(f"CUDA graph capture of the pricing step failed ({type(e).__name__}: {e}); running eagerly")
            self._capture_overcount += self.launches - launches
            self.use_graph = False
            torch.cuda.synchronize()
            return
        self._graph_launches = self.launches - launches
        self._capture_overcount += self._graph_launches       # recorded, not executed
        if self.fused:
            self.pricer._fused_passes -= 1
        self._graph = g

    def _read_result(self):
        K = max(self.K, 1)
        if self.world == 1:
            h = self.pricer.h_block.numpy()
            n_out = int(h[2 * K + 4]) if self.K > 0 else 0
            count, status = int(h[2 * K]) & 0xFFFFFFFFFFFFFFFF, int(h[2 * K + 3])
            res = dev.PriceResult(count, float(lib.sx_key_to_f64(int(h[2 * K + 1]))),
                                  h[K:K + n_out].copy(), h[:n_out].view(np.float64).copy())
            return res, status, count
        h = self.h_out.numpy()
        xs = int(h[2 * K + 5]) & 0xFFFFFFFF                    # int32 status word of the exchange / merge kernels
        if self.exchange in ("ll", "p2p") and xs:
            self._dead = True                                   # epochs may be out of step now (ADVICE r1)
            check(xs - (1 << 32) if xs >= (1 << 31) else xs, "peer exchange")
        n_out = int(h[2 * K]) if self.K > 0 else 0
        res = dev.PriceResult(int(h[2 * K + 1]), float(lib.sx_key_to_f64(int(h[2 * K + 2]))),
                              h[K:K + n_out].copy(), h[:n_out].view(np.float64).copy())
        return res, int(h[2 * K + 4]), int(h[2 * K + 3])

    def price(self, y_host: np.ndarray) -> dev.PriceResult:
        """One pass from a host vector of duals: copy into pinned memory, replay the captured step
        (H2D, pricing, selection, exchange + merge, D2H), one synchronisation, read the result."""
        if y_host is not self._h_y_np:                     # duals already written into `y_pinned`: nothing to copy
            r0 = self.row0
            self._h_y_np[r0:r0 + self.S_loc] = y_host[r0:r0 + self.S_loc]      # only what this rank uploads
            self._h_y_np[self.S:] = y_host[self.S:self.S + self.D]
        if self._graph is None and self.use_graph and not self._capture_tried:
            self._capture_tried = True
            self._capture()
        if self._dead:
            raise RuntimeError("this pricer saw a peer-exchange timeout; its epoch counters may be out of step with "
                               "the peers': build a new one")
        first = True
        while True:
            if first and self._graph is not None:
                self._graph.replay()
                self._replayed_launches += self._graph_launches
                if self.fused:
                    self.pricer.note_replayed_fused_passes(1)
            else:
                self._step()
            first = False
            torch.cuda.current_stream().synchronize()
            res, status, cmax = self._read_result()
            # Every rank reads the same folded status, so all ranks repeat the pass together, with a larger
            # candidate buffer after an overflow.
            res.status = status
            if self.K == 0 or (status & _native.SX_STATUS_CAND_OVERFLOW) == 0:
                return res
            self.pricer.grow(cmax)
            self._graph, self._capture_tried = None, False          # buffers moved: record again next time

    @property
    def y_pinned(self) -> np.ndarray:
        """The pinned host vector (S + D) that `price` uploads from.  Write the duals into it and pass this
        very array to `price` to skip the pageable-to-pinned copy."""
        return self._h_y_np

    @property
    def h2d_bytes(self):
        return 8 * (self.S_loc + self.D)

    @property
    def d2h_bytes(self):
        return 8 * (2 * max(self.K, 1) + 6)

"""Device-side operators of the hot path: thin wrappers that hand torch CUDA tensors
(device memory + the current stream; plumbing only) to the C ABI of libsxcross.

Every function fails loudly without a CUDA device or without the native library;
nothing here computes on the CPU.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass

import numpy as np
import torch

from . import _native
from ._native import check, lib

TOL_RC = 1e-6   # TOLERANCE_FOR_REDUCED_COSTS, reference parameters.py:8
FUSED_DEFAULT = True   # dense pricing passes use sx_price_dense_ot_fused when the matrix allows the TMA path


def _require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("smart_crossover device path needs a CUDA device (sm_100a); there is no CPU fallback")


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _ws(nbytes, device):
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


def _f64(t, device=None):
    """Contiguous float64 CUDA tensor from a tensor / ndarray."""
    _require_cuda()
    if isinstance(t, np.ndarray):
        t = torch.from_numpy(np.ascontiguousarray(t, dtype=np.float64))
    t = t.to(device=device or "cuda", dtype=torch.float64)
    return t.contiguous()


# ---- K1 ------------------------------------------------------------------------------------
def score_ot(x: torch.Tensor, s: torch.Tensor, d: torch.Tensor, want_hist: bool = False, out=None):
    """Flow indicators max(x_ij/s_i, x_ij/d_j); reference net_manager.py:377-378.  With want_hist also
    returns the 4096-bin histogram of the scores' top key bits (input of `kruskal_prefix`).  `out`: a
    contiguous S * D float64 tensor to write the scores into."""
    S, D = s.numel(), d.numel()
    out = torch.empty(S * D, dtype=torch.float64, device=x.device) if out is None else out
    hist = torch.zeros(4096, dtype=torch.int32, device=x.device) if want_hist else None
    check(lib.sx_score_ot(_ptr(x), _ptr(s), _ptr(d), S, D, _ptr(out), _ptr(hist), _stream()), "sx_score_ot")
    return (out, hist) if want_hist else out


def score_mcf(x, u, tail, head, node_ptr, node_arc, node_sign) -> torch.Tensor:
    """MCF flow indicators; reference net_manager.py:165-182."""
    N, E = node_ptr.numel() - 1, x.numel()
    out = torch.empty(E, dtype=torch.float64, device=x.device)
    ws = _ws(lib.sx_score_mcf_workspace_bytes(N, E), x.device)
    check(lib.sx_score_mcf(_ptr(x), _ptr(u), _ptr(tail), _ptr(head), _ptr(node_ptr), _ptr(node_arc),
                           _ptr(node_sign), N, E, _ptr(out), _ptr(ws), ws.numel(), _stream()), "sx_score_mcf")
    return out


def argsort_f64(key: torch.Tensor, want_sorted=True):
    """Stable ascending argsort (ties by ascending id). Returns (order uint32-as-int32 tensor, sorted keys)."""
    n = key.numel()
    order = torch.empty(n, dtype=torch.int32, device=key.device)   # holds uint32 bit patterns
    sorted_key = torch.empty(n, dtype=torch.float64, device=key.device) if want_sorted else None
    ws = _ws(lib.sx_argsort_workspace_bytes(n), key.device)
    check(lib.sx_argsort_f64(_ptr(key), n, _ptr(order), _ptr(sorted_key), _ptr(ws), ws.numel(), _stream()),
          "sx_argsort_f64")
    return order, sorted_key


def queue_from_order(order: torch.Tensor) -> torch.Tensor:
    """queue = argsort(score)[::-1] as int64; reference net_manager.py:184,379."""
    n = order.numel()
    q = torch.empty(n, dtype=torch.int64, device=order.device)
    check(lib.sx_queue_from_order(_ptr(order), n, _ptr(q), _stream()), "sx_queue_from_order")
    return q


def kruskal_order(sorted_key: torch.Tensor, order: torch.Tensor) -> torch.Tensor:
    """Descending key, ties by ascending id (SciPy Kruskal visiting order, tree_BI.py:47,53)."""
    n = order.numel()
    out = torch.empty(n, dtype=torch.int32, device=order.device)
    ws = _ws(lib.sx_kruskal_order_workspace_bytes(n), order.device)
    check(lib.sx_kruskal_order(_ptr(sorted_key), _ptr(order), n, _ptr(out), _ptr(ws), ws.numel(), _stream()),
          "sx_kruskal_order")
    return out


def kruskal_order_head(sorted_key: torch.Tensor, order: torch.Tensor, T: int, T_cap: int | None = None):
    """The first arcs of `kruskal_order` (at least T, whole tie runs) without flipping the whole array.
    Returns an int32 tensor or None when the tie runs at the cut hold more than T_cap arcs."""
    n = order.numel()
    T = int(min(T, n))
    T_cap = int(min(n, T_cap or max(2 * T, T + 65536)))
    out = torch.empty(T_cap, dtype=torch.int32, device=order.device)
    ws = _ws(lib.sx_kruskal_order_workspace_bytes(T_cap) + 256, order.device)
    n_head = ctypes.c_int64(0)
    check(lib.sx_kruskal_order_head(_ptr(sorted_key), _ptr(order), n, T, T_cap, _ptr(out), ctypes.byref(n_head),
                                    _ptr(ws), ws.numel(), _stream()), "sx_kruskal_order_head")
    if n_head.value < 0:
        return None
    return out[:n_head.value]


def kruskal_prefix(weights: torch.Tensor, T: int, T_cap: int | None = None, hist: torch.Tensor | None = None):
    """Head of the Kruskal order (descending weight, ties by ascending id): every arc at least as heavy
    as the T-th heaviest.  Returns an int32 tensor (uint32 bit patterns) or None when more than T_cap
    arcs tie at the threshold (the caller then sorts everything).  One stream synchronisation."""
    n = weights.numel()
    T = int(min(T, n))
    T_cap = int(T_cap or max(2 * T, T + 65536))
    out = torch.empty(T_cap, dtype=torch.int32, device=weights.device)
    ws = _ws(lib.sx_kruskal_prefix_workspace_bytes(T_cap), weights.device)
    n_prefix = ctypes.c_int64(0)
    check(lib.sx_kruskal_prefix(_ptr(weights), n, T, T_cap, _ptr(hist), _ptr(out), ctypes.byref(n_prefix), _ptr(ws),
                                ws.numel(), _stream()), "sx_kruskal_prefix")
    if n_prefix.value < 0:
        return None
    return out[:n_prefix.value]


# ---- K2 ------------------------------------------------------------------------------------
def kruskal(korder: torch.Tensor, N: int, S: int = 0, D: int = 0, tail=None, head=None):
    """Spanning forest over `korder`; returns (tree arc ids ascending [device, capacity N-1], n_tree [device])."""
    n = korder.numel()
    tree = torch.empty(max(N - 1, 1), dtype=torch.int64, device=korder.device)
    n_tree = torch.zeros(1, dtype=torch.int64, device=korder.device)
    ws = _ws(lib.sx_kruskal_workspace_bytes(N, n), korder.device)
    check(lib.sx_kruskal(_ptr(korder), n, _ptr(tail), _ptr(head), S, D, N, _ptr(tree), _ptr(n_tree),
                         _ptr(ws), ws.numel(), _stream()), "sx_kruskal")
    return tree, n_tree


# ---- K3 ------------------------------------------------------------------------------------
def tree_potentials(tree: torch.Tensor, n_tree: int, N: int, cost: torch.Tensor, root: int, S: int = 0,
                    D: int = 0, ld: int = 0, tail=None, head=None, plus=_native.SX_PLUS_IS_HEAD) -> torch.Tensor:
    """y with y[root] = 0 and y[plus] - y[minus] = cost on every tree arc (SURVEY.md section 8 row a5).
    Raises SxError(SX_ERR_NOT_SPANNING) if the arcs are not a spanning tree."""
    y = torch.zeros(N, dtype=torch.float64, device=cost.device)
    status = torch.zeros(1, dtype=torch.int32, device=cost.device)
    ws = _ws(lib.sx_tree_potentials_workspace_bytes(N), cost.device)
    check(lib.sx_tree_potentials(_ptr(tree), n_tree, _ptr(tail), _ptr(head), S, D, N, _ptr(cost), ld or D,
                                 plus, root, _ptr(y), _ptr(status), _ptr(ws), ws.numel(), _stream()),
          "sx_tree_potentials")
    check(int(status.item()), "sx_tree_potentials")
    return y


def tree_flows(tree: torch.Tensor, n_tree: int, N: int, b: torch.Tensor, root: int, S: int = 0, D: int = 0,
               tail=None, head=None, plus=_native.SX_PLUS_IS_HEAD) -> torch.Tensor:
    """Primal flows x_T of the tree basis, B x_T = b[:-1] (reference tree_BI.py:74-76), one per tree arc."""
    flow = torch.zeros(max(n_tree, 1), dtype=torch.float64, device=b.device)
    status = torch.zeros(1, dtype=torch.int32, device=b.device)
    ws = _ws(lib.sx_tree_potentials_workspace_bytes(N), b.device)
    check(lib.sx_tree_flows(_ptr(tree), n_tree, _ptr(tail), _ptr(head), S, D, N, _ptr(b), plus, root,
                            _ptr(flow), _ptr(status), _ptr(ws), ws.numel(), _stream()), "sx_tree_flows")
    check(int(status.item()), "sx_tree_flows")
    return flow[:n_tree]


# ---- K4 ------------------------------------------------------------------------------------
@dataclass
class PriceResult:
    n_violating: int
    min_rc: float
    topk_id: np.ndarray     # int64, ascending (rc, id)
    topk_rc: np.ndarray     # float64
    rc: torch.Tensor | None = None   # full reduced costs if requested (device)
    status: int = 0                  # SX_STATUS_* bits of the pass (SX_STATUS_NAN_RC: some reduced cost was NaN)

    @property
    def has_nan(self) -> bool:
        return bool(self.status & _native.SX_STATUS_NAN_RC)

    @property
    def optimal(self) -> bool:
        """`np.all(rc >= -tol)` (net_manager.py:318,496): no violator and no NaN reduced cost."""
        return self.n_violating == 0 and not self.has_nan


class Pricer:
    """Reusable buffers for repeated pricing passes over one problem (one CG loop).

    The top-K rc list, the id list, the pricing header and the output count live in ONE int64
    tensor `block = [K rc bits | K ids | header (4) | n_out | pad]`, so a rank's whole contribution
    to the multi-GPU exchange -- and the per-pass read-back -- is a single contiguous buffer."""

    BLOCK_TAIL = 6      # header (4) + n_out + pad (block length stays even: 16-byte peer stores)

    def __init__(self, device, K: int, cand_cap: int | None = None, fused: bool | None = None):
        _require_cuda()
        self.device = device
        self.K = int(K)
        if cand_cap is None:
            cand_cap = max(64 * self.K, 1 << 20) if self.K > 0 else 0
        self.cap = int(cand_cap)
        self.sel = torch.zeros(lib.sx_select_state_bytes(), dtype=torch.uint8, device=device) if self.K > 0 else None
        self._alloc()
        Kp = max(self.K, 1)
        self.Kp = Kp
        self.block = torch.zeros(2 * Kp + self.BLOCK_TAIL, dtype=torch.int64, device=device)
        self.out_rc = self.block[:Kp].view(torch.float64)
        self.out_id = self.block[Kp:2 * Kp]
        self.header = self.block[2 * Kp:2 * Kp + 4]
        self.out_n = self.block[2 * Kp + 4:2 * Kp + 5]
        # pinned staging for the per-pass host round trip
        self.h_block = torch.zeros(2 * Kp + self.BLOCK_TAIL, dtype=torch.int64).pin_memory()
        self.launches = 0
        # fused pass (sx_price_dense_ot_fused): two selection states used by alternate passes + control block
        self.fused = bool(FUSED_DEFAULT if fused is None else fused) and Kp <= _native.SX_TOPK_MAX_K
        self._fused_passes, self._last_fused = 0, False
        if self.fused:
            self.fstate = torch.zeros(lib.sx_fused_state_bytes(), dtype=torch.uint8, device=device)
            check(lib.sx_fused_state_init(_ptr(self.fstate), Kp, _stream()), "sx_fused_state_init")

    def _alloc(self):
        self.cand_rc = torch.empty(max(self.cap, 1), dtype=torch.float64, device=self.device)
        self.cand_id = torch.empty(max(self.cap, 1), dtype=torch.int64, device=self.device)
        self.ws = _ws(lib.sx_topk_workspace_bytes(self.cap, max(self.K, 1)), self.device)

    def reset(self):
        check(lib.sx_price_pass_begin(_ptr(self.header), _ptr(self.sel), self.K, _stream()), "sx_price_pass_begin")
        self.launches += 1
        self._last_fused = False

    def price_dense(self, M, ld, row0, S_loc, D, y_src, y_dst, tol=TOL_RC, rc_out=None, variant=-1):
        check(lib.sx_price_dense_ot(_ptr(M), ld, row0, S_loc, D, _ptr(y_src), _ptr(y_dst), float(tol),
                                    _ptr(self.header), _ptr(self.sel), _ptr(self.cand_rc), _ptr(self.cand_id),
                                    self.cap if self.K > 0 else 0, _ptr(rc_out), D if rc_out is not None else 0,
                                    variant, _stream()),
              "sx_price_dense_ot")
        self.launches += 1

    @staticmethod
    def fusable(M, ld) -> bool:
        """The fused pass needs the TMA path: 16-byte aligned base and an even leading dimension."""
        return M.data_ptr() % 16 == 0 and ld % 2 == 0

    def price_dense_fused(self, M, ld, row0, S_loc, D, y_src, y_dst, tol=TOL_RC, peer_bufs=None, rank=0, G=1,
                          merged=None, xstatus=None, lb=None, bigm=None):
        """begin + pricing + selection (+ push of the block to `peer_bufs`, + merge of the G blocks into
        `merged`) as one launch.  `lb`: the lower-bound copy of M (`cost_lb`); the pass may then stream it
        instead of M, with the same results.  `bigm` = (S, y_art, bigM, corner): price the slab as rows
        [row0, row0 + S_loc) of the (S+1) x (D+1) big-M extension of an S x D base (`sx_price_dense_ot_fused_bigm`):
        y_dst then holds D + 1 sink duals, y_art (device, one element) is u_S, and ids are the extension's."""
        if bigm is not None:
            S, y_art, bigM, corner = bigm
            check(lib.sx_price_dense_ot_fused_bigm(_ptr(M), ld, _ptr(lb), lb.stride(0) if lb is not None else 0, row0,
                                                   S_loc, S, D, _ptr(y_src), _ptr(y_dst), _ptr(y_art), float(bigM),
                                                   float(corner), float(tol), _ptr(self.fstate), _ptr(self.cand_rc),
                                                   _ptr(self.cand_id), self.cap if self.K > 0 else 0, self.Kp,
                                                   _ptr(self.block), self.block.numel(), peer_bufs, rank, G,
                                                   _ptr(merged), _ptr(xstatus), _ptr(self.ws), self.ws.numel(),
                                                   _stream()), "sx_price_dense_ot_fused_bigm")
        elif lb is not None:
            check(lib.sx_price_dense_ot_fused_lb(_ptr(M), ld, _ptr(lb), lb.stride(0), row0, S_loc, D, _ptr(y_src),
                                                 _ptr(y_dst), float(tol), _ptr(self.fstate), _ptr(self.cand_rc),
                                                 _ptr(self.cand_id), self.cap if self.K > 0 else 0, self.Kp,
                                                 _ptr(self.block), self.block.numel(), peer_bufs, rank, G, _ptr(merged),
                                                 _ptr(xstatus), _ptr(self.ws), self.ws.numel(), _stream()),
                  "sx_price_dense_ot_fused_lb")
        else:
            check(lib.sx_price_dense_ot_fused(_ptr(M), ld, row0, S_loc, D, _ptr(y_src), _ptr(y_dst), float(tol),
                                              _ptr(self.fstate), _ptr(self.cand_rc), _ptr(self.cand_id),
                                              self.cap if self.K > 0 else 0, self.Kp, _ptr(self.block),
                                              self.block.numel(), peer_bufs, rank, G, _ptr(merged), _ptr(xstatus),
                                              _ptr(self.ws), self.ws.numel(), _stream()), "sx_price_dense_ot_fused")
        self.launches += 1
        self._fused_passes += 1
        self._last_fused = True

    def fused_phase_us(self):
        """Where CTA 0 of the last fused pass spent its time (us): pricing, barrier 1, filter, barrier 2, rank."""
        off = lib.sx_fused_state_timestamps_offset()
        t = self.fstate[off:off + 64].view(torch.int64).cpu().numpy()
        names = ["pricing", "barrier1", "bound+filter", "barrier2", "rank+emit"]
        out = {n: round(float(t[i + 1] - t[i]) * 1e-3, 2) for i, n in enumerate(names)}
        out["last_cta_end_(after_merge_if_any)_minus_cta0_rank_end"] = round(float(t[6] - t[5]) * 1e-3, 2)
        out["gap_since_previous_pass_end"] = round(float(t[0] - t[7]) * 1e-3, 2)
        return out

    def fused_walk(self) -> int:
        """What the last fused pass streamed: 1 = the lower-bound copy, 0 = M itself (diagnostics; synchronises)."""
        off = lib.sx_fused_state_timestamps_offset() - 12
        return int(self.fstate[off:off + 4].view(torch.int32).item())

    def note_replayed_fused_passes(self, n: int = 1):
        """A captured CUDA graph holding a fused pass was replayed n times (keeps `n_candidates` right)."""
        self._fused_passes += n

    def n_candidates(self) -> int:
        """Length of the (pruned) candidate list the last pass left (diagnostics / tests); synchronises."""
        if self.K == 0:
            return 0
        if self._last_fused:
            off = ((self._fused_passes - 1) & 1) * lib.sx_select_state_bytes()
            return int(self.fstate[off:off + 8].view(torch.int64).item())
        return int(self.sel[:8].view(torch.int64).item())

    def price_arcs(self, c, tail, head, vbasis, y, id0=0, tol=TOL_RC, rc_out=None):
        check(lib.sx_price_arcs(_ptr(c), _ptr(tail), _ptr(head), _ptr(vbasis), _ptr(y), c.numel(), id0,
                                float(tol), _ptr(self.header), _ptr(self.sel), _ptr(self.cand_rc),
                                _ptr(self.cand_id), self.cap if self.K > 0 else 0, _ptr(rc_out), _stream()),
              "sx_price_arcs")
        self.launches += 1

    def select(self):
        """Enqueue the top-K selection over the candidates (device only)."""
        if self.K > 0:
            check(lib.sx_topk_select(_ptr(self.cand_rc), _ptr(self.cand_id), self.cap, _ptr(self.sel),
                                     _ptr(self.header), self.K, _ptr(self.out_rc), _ptr(self.out_id),
                                     _ptr(self.out_n), _ptr(self.ws), self.ws.numel(), _stream()), "sx_topk_select")
            self.launches += 6 if self.K > _native.SX_TOPK_MAX_K else 2

    def fetch(self) -> PriceResult:
        """Device -> pinned host copy of the block (top-K + header + count); one synchronisation."""
        self.h_block.copy_(self.block, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        h = self.h_block.numpy()
        Kp = self.Kp
        self.status = int(h[2 * Kp + 3])
        if self.status & _native.SX_STATUS_K_MISMATCH:
            raise ValueError("top-k selection asked for more arcs than the pricing pass was started for")
        if self.status & _native.SX_STATUS_DUPLICATE_CANDIDATES:
            raise ValueError("top-k selection found one arc priced into the pass many times: "
                             "a pass must price every arc at most once")
        nviol = int(h[2 * Kp]) & 0xFFFFFFFFFFFFFFFF
        min_rc = float(lib.sx_key_to_f64(int(h[2 * Kp + 1])))
        k = int(h[2 * Kp + 4]) if self.K > 0 else 0
        return PriceResult(nviol, min_rc, h[Kp:Kp + k].copy(), h[:k].view(np.float64).copy(), status=self.status)

    def overflowed(self, res: PriceResult | None = None) -> bool:
        return self.K > 0 and bool(self.status & _native.SX_STATUS_CAND_OVERFLOW)

    MAX_CAP = 1 << 28      # 256 M candidates (4 GB + 8 GB of selection lists): beyond this the pass cannot be pruned

    def grow(self, n_violating: int = 0):
        """Enlarge the candidate buffer after SX_STATUS_CAND_OVERFLOW (x4, at most every violator)."""
        if self.cap >= self.MAX_CAP:
            raise RuntimeError("pricing candidates cannot be pruned below %d entries: more arcs than that tie "
                               "(to 0.4 %%) with the K-th most violating one" % self.MAX_CAP)
        self.cap = min(max(4 * self.cap, 1024), self.MAX_CAP)
        if n_violating:
            self.cap = min(self.cap, max(int(n_violating), 1024))
        self._alloc()


def price_dense_ot(M: torch.Tensor, y: torch.Tensor, K: int = 0, tol: float = TOL_RC, want_rc=False,
                   variant=-1, pricer: Pricer | None = None, fused: bool | None = None) -> PriceResult:
    """One pricing pass over a device-resident S x D cost matrix with duals y (S + D).
    rc_ij = M_ij - (y[S+j] - y[i]); reference net_manager.py:474-497."""
    S, D = M.shape
    pr = pricer or Pricer(M.device, K, fused=(FUSED_DEFAULT if fused is None else fused) and not want_rc
                          and variant in (-1, 0))
    rc = torch.empty(S * D, dtype=torch.float64, device=M.device) if want_rc else None
    fused = pr.fused and fused is not False and not want_rc and variant in (-1, 0) \
        and Pricer.fusable(M, M.stride(0)) and S > 0
    while True:
        if fused:
            pr.price_dense_fused(M, M.stride(0), 0, S, D, y[:S], y[S:S + D], tol)
        else:
            pr.reset()
            pr.price_dense(M, M.stride(0), 0, S, D, y[:S], y[S:S + D], tol, rc, variant)
            pr.select()
        res = pr.fetch()
        if not pr.overflowed(res):
            break
        pr.grow(res.n_violating)       # more violators than candidate slots: size exactly, price again
    res.rc = rc
    return res


def price_arcs(c, tail, head, y, vbasis=None, K: int = 0, tol: float = TOL_RC, want_rc=False,
               pricer: Pricer | None = None) -> PriceResult:
    """Arc-list pricing rc_k = c_k - (y[tail_k] - y[head_k]), negated where vbasis == -2;
    reference net_manager.py:293-319."""
    pr = pricer or Pricer(c.device, K)
    rc = torch.empty(c.numel(), dtype=torch.float64, device=c.device) if want_rc else None
    while True:
        pr.reset()
        pr.price_arcs(c, tail, head, vbasis, y, 0, tol, rc)
        pr.select()
        res = pr.fetch()
        if not pr.overflowed(res):
            break
        pr.grow(res.n_violating)
    res.rc = rc
    return res


def topk_merge(blocks_rc: torch.Tensor, blocks_id: torch.Tensor, headers: torch.Tensor | None = None):
    """Merge G sorted, padded top-K lists into one (rc, id, n[, summary]) on the device.

    blocks_rc / blocks_id are (G, K) views that may be strided (e.g. columns of the all-gathered
    (G, 2K+4) buffer); `headers` (G, 4) with the same row stride folds the per-rank
    pricing headers into summary = {total, min key, largest single count, OR of status words}."""
    G, K = blocks_rc.shape
    stride = blocks_rc.stride(0)
    assert blocks_id.stride(0) == stride and blocks_rc.stride(1) == 1 and blocks_id.stride(1) == 1
    dev_ = blocks_rc.device
    out_rc = torch.empty(K, dtype=torch.float64, device=dev_)
    out_id = torch.empty(K, dtype=torch.int64, device=dev_)
    out_n = torch.zeros(1, dtype=torch.int64, device=dev_)
    summary = torch.zeros(4, dtype=torch.int64, device=dev_) if headers is not None else None
    if headers is not None:
        assert headers.stride(0) == stride
    ws = _ws(lib.sx_topk_merge_workspace_bytes(G), dev_)
    check(lib.sx_topk_merge(_ptr(blocks_rc), _ptr(blocks_id), stride, G, K, _ptr(headers), _ptr(out_rc),
                            _ptr(out_id), _ptr(out_n), _ptr(summary), None, 0, _ptr(ws), ws.numel(), _stream()),
          "sx_topk_merge")
    if headers is not None:
        return out_rc, out_id, out_n, summary
    return out_rc, out_id, out_n


def cost_lb(M: torch.Tensor) -> torch.Tensor:
    """Lower-bound copy of a device cost matrix for the fused pass (`sx_cost_lb_build`): the high 32 bits of each
    fp64 cost rounded toward -inf (int32 bit patterns; as the high half of a double they are <= M element by
    element), row stride a multiple of 4 words.  Raises torch.OutOfMemoryError when it does not fit."""
    S, D = M.shape
    ld_lb = (D + 3) // 4 * 4
    lb = torch.empty(S, ld_lb, dtype=torch.int32, device=M.device)
    check(lib.sx_cost_lb_build(_ptr(M), M.stride(0), S, D, _ptr(lb), ld_lb, _stream()), "sx_cost_lb_build")
    return lb


# ---- persistent, row-sharded pricer behind the managers (sx_ot_pricer) --------------------------------
MIN_ARCS_PER_DEVICE = 1 << 25      # below ~3e7 arcs (270 MB) per GPU another device only adds latency


def pricing_devices(n_arcs: int, S: int) -> list:
    """Devices a dense OT problem of n_arcs is priced on: `SX_DEVICES` ("all", a count or a comma list) or
    as many visible GPUs as give each at least MIN_ARCS_PER_DEVICE arcs, starting at the current device."""
    import os
    _require_cuda()
    n_vis, cur = torch.cuda.device_count(), torch.cuda.current_device()
    spec = os.environ.get("SX_DEVICES", "").strip()
    if spec and spec != "all" and "," in spec:
        devs = [int(v) for v in spec.split(",")]
    else:
        want = n_vis if spec == "all" else (int(spec) if spec else max(1, n_arcs // MIN_ARCS_PER_DEVICE))
        devs = [(cur + i) % n_vis for i in range(max(1, min(want, n_vis)))]
    devs = devs[:max(1, min(len(devs), S))]
    if len(devs) > 1 and not all(torch.cuda.can_device_access_peer(a, b) for a in devs for b in devs if a != b):
        devs = devs[:1]
    return devs


def balanced_row_bounds(S: int, seconds_per_row, multiple: int = 16):
    """Row partition with shares proportional to each shard's measured rate (1 / seconds per row), boundaries
    rounded to a multiple of the pricing kernel's 16-row tiles.  A pass ends when the slowest GPU has delivered
    its block, and the GPUs of one box stream at rates a few percent apart."""
    rate = 1.0 / np.asarray(seconds_per_row, dtype=np.float64)
    cum = np.concatenate([[0.0], np.cumsum(rate)]) / rate.sum() * S
    b = [int(round(v / multiple) * multiple) for v in cum]
    b[0], b[-1] = 0, int(S)
    for g in range(1, len(b)):                      # keep every shard non-empty
        b[g] = max(b[g], b[g - 1] + 1) if g < len(b) - 1 else b[g]
    for g in range(len(b) - 2, 0, -1):
        b[g] = min(b[g], b[g + 1] - 1)
    return b


class CostSlabs:
    """Row shards of a dense S x D matrix, one per device, resident for the life of the problem (as the
    reference keeps `ot.M` in its manager).  A cost matrix has its leading dimension rounded up to even (TMA
    path); a flow or its scores (`pad_ld=False`) has contiguous rows, which `sx_score_ot` needs."""

    def __init__(self, S: int, D: int, devices, row_bounds=None, pad_ld: bool = True):
        """`row_bounds` (G + 1 increasing row indices from 0 to S): shard g = rows [row_bounds[g], row_bounds[g+1]);
        default = equal shares.  See `balanced_row_bounds`."""
        _require_cuda()
        self.S, self.D, self.devices = int(S), int(D), list(devices)
        self.ld = self.D + (self.D & 1) if pad_ld else self.D
        G = len(self.devices)
        if row_bounds is None:
            row_bounds = [self.S * g // G for g in range(G + 1)]
        row_bounds = [int(v) for v in row_bounds]
        if len(row_bounds) != G + 1 or row_bounds[0] != 0 or row_bounds[-1] != self.S \
                or any(b <= a for a, b in zip(row_bounds, row_bounds[1:])):
            raise ValueError("row_bounds must be G + 1 strictly increasing row indices from 0 to S")
        self.row_bounds = row_bounds
        self.row0 = row_bounds[:-1]
        self.rows = [row_bounds[g + 1] - row_bounds[g] for g in range(G)]
        self.t = [torch.empty(self.rows[g], self.ld, dtype=torch.float64, device=torch.device("cuda", d))
                  for g, d in enumerate(self.devices)]

    def view(self, g: int) -> torch.Tensor:
        """(rows_g, D) view of shard g."""
        return self.t[g][:, :self.D]

    def max(self) -> float:
        """Largest entry of the S x D matrix over every shard (not the `ld` padding); NaN if any entry is NaN, as
        `np.max` gives."""
        return float(np.max([torch.amax(self.view(g)).item() for g in range(len(self.devices))]))

    def same_shards(self, other: "CostSlabs") -> bool:
        """Whether `other` has this matrix's shape, devices and row bounds."""
        return (self.S, self.D, self.devices, self.row_bounds) == (other.S, other.D, other.devices, other.row_bounds)

    def take_flat(self, ids) -> np.ndarray:
        """Entries at row-major ids (host int64 array), gathered shard by shard on the devices."""
        ids = np.asarray(ids, dtype=np.int64)
        out = np.empty(ids.shape)
        i, j = np.divmod(ids, self.D)
        for g, d in enumerate(self.devices):
            r0, rows = self.row0[g], self.rows[g]
            m = (i >= r0) & (i < r0 + rows)
            if m.any():
                ii = torch.from_numpy(i[m] - r0).to(torch.device("cuda", d))
                jj = torch.from_numpy(j[m]).to(torch.device("cuda", d))
                out[m] = self.t[g][ii, jj].cpu().numpy()
        return out

    @classmethod
    def from_host(cls, M, devices=None, border=None, row_bounds=None, like: "CostSlabs | None" = None):
        """Upload a host matrix.  `border` = (bigM, corner): the device matrix is the (S+1) x (D+1) big-M
        extension of M (net_manager.py:390-393) -- last row / column = bigM, corner = `corner` -- built on the
        device, so the extended matrix never exists on the host.  `like`: a flow (S x D, or S * D flat) for the
        problem whose cost slabs `like` are -- same devices and row bounds, contiguous rows."""
        M = np.asarray(M, dtype=np.float64)
        if like is not None:
            M = M.reshape(like.S, like.D)
        S0, D0 = M.shape
        S, D = (S0 + 1, D0 + 1) if border is not None else (S0, D0)
        if like is not None:
            self = cls(S, D, like.devices, like.row_bounds, pad_ld=False)
        else:
            self = cls(S, D, devices, row_bounds)
        for g in range(len(self.devices)):
            r0, r1 = self.row0[g], self.row0[g] + self.rows[g]
            h1 = min(r1, S0)
            if h1 > r0:                                        # rows of M in this shard (staged upload when large)
                self.t[g][:h1 - r0, :D0].copy_(to_device(M[r0:h1], device=self.t[g].device))
            if border is not None:
                self.t[g][:, D0] = float(border[0])
                if r1 == S:                                    # the artificial source is the last row
                    self.t[g][-1, :D0] = float(border[0])
                    self.t[g][-1, D0] = float(border[1])
        self.sync()
        return self

    def sync(self):
        for d in self.devices:
            torch.cuda.synchronize(d)


class OTPricer:
    """`sx_ot_pricer`: persistent pricer of one dense OT problem over the devices of its `CostSlabs`.
    `price(y_src, y_dst)` takes HOST vectors (the LP solver's duals) and returns a PriceResult; nothing is
    allocated per pass.  One kernel per GPU and pass (price + select + NVLink push + merge).

    `bigm` = (bigM, corner): the slabs are the S x D base of a problem extended by big-M, and the pricer prices the
    (S+1) x (D+1) extension (`sx_ot_pricer_create_bigm`; the extended matrix is never built): `price` takes S + 1
    and D + 1 duals and returns arc ids of the extension."""

    def __init__(self, slabs: CostSlabs, K: int, tol: float = TOL_RC, bigm=None):
        _require_cuda()
        self.slabs, self.K = slabs, int(K)
        self.bigm = None if bigm is None else (float(bigm[0]), float(bigm[1]))
        G = len(slabs.devices)
        devs = (ctypes.c_int * G)(*slabs.devices)
        ptrs = (ctypes.c_void_p * G)(*[t.data_ptr() for t in slabs.t])
        self._h = ctypes.c_void_p()
        slabs.sync()
        bounds = (ctypes.c_int64 * (G + 1))(*slabs.row_bounds)
        if self.bigm is None:
            check(lib.sx_ot_pricer_create(G, devs, ptrs, bounds, slabs.ld, slabs.S, slabs.D, self.K, float(tol),
                                          ctypes.byref(self._h)), "sx_ot_pricer_create")
        else:
            check(lib.sx_ot_pricer_create_bigm(G, devs, ptrs, bounds, slabs.ld, slabs.S, slabs.D, self.bigm[0],
                                               self.bigm[1], self.K, float(tol), ctypes.byref(self._h)),
                  "sx_ot_pricer_create_bigm")
        Kp = max(self.K, 1)
        self._rc = np.empty(Kp, dtype=np.float64)
        self._id = np.empty(Kp, dtype=np.int64)
        self._cnt, self._min = ctypes.c_ulonglong(0), ctypes.c_double(0.0)
        self._n, self._status = ctypes.c_int64(0), ctypes.c_ulonglong(0)

    def price(self, y_src: np.ndarray, y_dst: np.ndarray) -> PriceResult:
        y_src = np.ascontiguousarray(y_src, dtype=np.float64)
        y_dst = np.ascontiguousarray(y_dst, dtype=np.float64)
        ext = 1 if self.bigm is not None else 0
        if y_src.size != self.slabs.S + ext or y_dst.size != self.slabs.D + ext:
            raise ValueError("dual vectors do not match the cost matrix")
        check(lib.sx_ot_pricer_price_h(self._h, y_src.ctypes.data, y_dst.ctypes.data, ctypes.byref(self._cnt),
                                       ctypes.byref(self._min), self._rc.ctypes.data, self._id.ctypes.data,
                                       ctypes.byref(self._n), ctypes.byref(self._status)), "sx_ot_pricer_price_h")
        k = int(self._n.value) if self.K > 0 else 0
        return PriceResult(int(self._cnt.value), float(self._min.value), self._id[:k].copy(), self._rc[:k].copy(),
                           status=int(self._status.value))

    def stats(self) -> dict:
        a, b = ctypes.c_ulonglong(0), ctypes.c_ulonglong(0)
        f, m = ctypes.c_int(0), ctypes.c_int(0)
        check(lib.sx_ot_pricer_stats(self._h, ctypes.byref(a), ctypes.byref(b), ctypes.byref(f), ctypes.byref(m)),
              "sx_ot_pricer_stats")
        return {"passes": a.value, "repeated_passes": b.value, "fused": bool(f.value), "merge_in_kernel": bool(m.value),
                "devices": list(self.slabs.devices)}

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib.sx_ot_pricer_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def score_ot_slabs(x: CostSlabs, s: np.ndarray, d: np.ndarray):
    """`score_ot` on every shard of a row-sharded flow, each on its own device: (score slabs with x's devices and
    row bounds, each shard's level-0 histogram).  The scores never leave their devices."""
    if x.ld != x.D:
        raise ValueError("a sharded flow needs contiguous rows (CostSlabs(..., pad_ld=False) / from_host(like=))")
    s = np.ascontiguousarray(s, dtype=np.float64)
    d = np.ascontiguousarray(d, dtype=np.float64)
    if s.size != x.S or d.size != x.D:
        raise ValueError("marginals do not match the flow")
    out = CostSlabs(x.S, x.D, x.devices, x.row_bounds, pad_ld=False)
    hists = []
    for g, dv in enumerate(x.devices):
        with torch.cuda.device(dv):
            r0 = x.row0[g]
            s_g = torch.from_numpy(s[r0:r0 + x.rows[g]]).cuda()
            d_g = torch.from_numpy(d).cuda()
            hists.append(score_ot(x.t[g], s_g, d_g, want_hist=True, out=out.t[g].view(-1))[1])
    return out, hists


def order_head_sharded(w: CostSlabs, T: int, T_cap: int | None = None, hists=None, queue: bool = False):
    """Head of the order of row-sharded weights (`sx_order_head_sharded_h`), on w.devices[0]: queue=False gives the
    Kruskal order (descending weight, ties by ascending id; int32 tensor of uint32 ids), queue=True the queue order
    (descending weight, ties by descending id; int64).  At least min(T, n) arcs, whole tie runs; None when more
    than T_cap arcs tie at the threshold.  `hists`: the shards' level-0 histograms (`score_ot_slabs`)."""
    if w.ld != w.D:
        raise ValueError("sharded weights need contiguous rows")
    G, n = len(w.devices), w.S * w.D
    T = int(min(T, n))
    T_cap = int(min(n, T_cap or max(2 * T, T + 65536)))
    d0 = torch.device("cuda", w.devices[0])
    out = torch.empty(T_cap, dtype=torch.int64 if queue else torch.int32, device=d0)
    w.sync()                      # the weights (and `out`'s memory) are ready before the library's own streams run
    hist_ptrs = (ctypes.c_void_p * G)(*[h.data_ptr() for h in hists]) if hists is not None else None
    n_out = ctypes.c_int64(0)
    check(lib.sx_order_head_sharded_h(G, (ctypes.c_int * G)(*w.devices),
                                      (ctypes.c_void_p * G)(*[t.data_ptr() for t in w.t]),
                                      (ctypes.c_int64 * (G + 1))(*w.row_bounds), w.S, w.D, T, T_cap, hist_ptrs,
                                      _native.SX_ORDER_QUEUE if queue else _native.SX_ORDER_KRUSKAL, _ptr(out),
                                      ctypes.byref(n_out)), "sx_order_head_sharded_h")
    if n_out.value < 0:
        return None
    return out[:n_out.value]


# ---- large device -> host downloads (get_sorted_flows returns two n-sized NumPy arrays) -----------------
_STAGE_BYTES = 32 << 20
_stage = {}          # device index -> (pinned staging buffers, copy stream, thread pool)


def to_host(t: torch.Tensor, ready: "torch.cuda.Event | None" = None) -> np.ndarray:
    """Contiguous device tensor -> fresh (pageable) NumPy array.  Above 64 MB the copy goes through four pinned
    32 MB staging buffers on a copy stream, and the pinned -> pageable copies run on a small thread pool while
    the next chunks are in flight: a plain `tensor.cpu()` of pageable memory is one thread's memcpy behind a
    serial DMA (~0.25 s for the 3.2 GB of scores at 20 000 x 20 000, more than every kernel of the path).
    `ready`: event after which `t` is complete; the copy stream then waits for it only, not for everything
    enqueued on the current stream since (the sort that follows the scores runs while they download)."""
    t = t.contiguous()
    nbytes = t.numel() * t.element_size()
    if nbytes < (64 << 20):
        return t.cpu().numpy()        # (synchronises the current stream; small enough not to matter)
    from concurrent.futures import ThreadPoolExecutor
    dev_index = t.device.index if t.device.index is not None else torch.cuda.current_device()
    if dev_index not in _stage:
        bufs = [torch.empty(_STAGE_BYTES, dtype=torch.uint8).pin_memory() for _ in range(4)]
        _stage[dev_index] = (bufs, torch.cuda.Stream(device=t.device), ThreadPoolExecutor(max_workers=4))
    bufs, stream, pool = _stage[dev_index]
    src = t.view(torch.uint8).reshape(-1) if t.dtype != torch.uint8 else t.reshape(-1)
    out = np.empty(t.shape, dtype=torch.empty(0, dtype=t.dtype).numpy().dtype)
    out_b = out.reshape(-1).view(np.uint8)
    if ready is not None:
        stream.wait_event(ready)
    else:
        stream.wait_stream(torch.cuda.current_stream(t.device))
    pending = [None] * len(bufs)               # per staging buffer: (event of its DMA, future of its host copy)
    n_chunks = (nbytes + _STAGE_BYTES - 1) // _STAGE_BYTES

    def drain(lo, hi, buf, ev):
        ev.synchronize()
        np.copyto(out_b[lo:hi], buf[:hi - lo].numpy())

    with torch.cuda.stream(stream):
        for i in range(n_chunks):
            b = i % len(bufs)
            if pending[b] is not None:
                pending[b].result()            # the buffer's previous chunk has left it
            lo, hi = i * _STAGE_BYTES, min(nbytes, (i + 1) * _STAGE_BYTES)
            bufs[b][:hi - lo].copy_(src[lo:hi], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(stream)
            pending[b] = pool.submit(drain, lo, hi, bufs[b], ev)
    for f in pending:
        if f is not None:
            f.result()
    t.record_stream(stream)
    return out


def to_device(a: np.ndarray, device=None, dtype=None) -> torch.Tensor:
    """NumPy array -> device tensor; above 64 MB through the same pinned staging buffers as `to_host`, the
    pageable -> pinned copies on the thread pool (the flow x of a 20 000 x 20 000 problem is 3.2 GB)."""
    _require_cuda()
    a = np.ascontiguousarray(a)
    device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if a.nbytes < (64 << 20) or (dtype is not None and torch.empty(0, dtype=dtype).numpy().dtype != a.dtype):
        t = torch.from_numpy(a)
        return (t.to(dtype) if dtype is not None else t).to(device)
    from concurrent.futures import ThreadPoolExecutor
    dev_index = device.index if device.index is not None else torch.cuda.current_device()
    if dev_index not in _stage:
        bufs = [torch.empty(_STAGE_BYTES, dtype=torch.uint8).pin_memory() for _ in range(4)]
        _stage[dev_index] = (bufs, torch.cuda.Stream(device=device), ThreadPoolExecutor(max_workers=4))
    bufs, stream, pool = _stage[dev_index]
    out = torch.empty(a.shape, dtype=torch.from_numpy(a[:0].reshape(-1)).dtype, device=device)
    dst = out.view(torch.uint8).reshape(-1)
    src = a.reshape(-1).view(np.uint8)
    nbytes = a.nbytes
    n_chunks = (nbytes + _STAGE_BYTES - 1) // _STAGE_BYTES
    events = [None] * len(bufs)
    fill = lambda lo, hi, buf: np.copyto(buf[:hi - lo].numpy(), src[lo:hi])
    futs = {}
    look = len(bufs) - 1                       # chunks whose host copy runs ahead of the DMA
    stream.wait_stream(torch.cuda.current_stream(device))
    with torch.cuda.stream(stream):
        for i in range(n_chunks + look):
            if i < n_chunks:                   # start filling buffer i % 4 once its previous DMA is done
                b = i % len(bufs)
                if events[b] is not None:
                    events[b].synchronize()
                lo, hi = i * _STAGE_BYTES, min(nbytes, (i + 1) * _STAGE_BYTES)
                futs[i] = pool.submit(fill, lo, hi, bufs[b])
            j = i - look
            if j >= 0:                         # DMA of chunk j
                futs.pop(j).result()
                b = j % len(bufs)
                lo, hi = j * _STAGE_BYTES, min(nbytes, (j + 1) * _STAGE_BYTES)
                dst[lo:hi].copy_(bufs[b][:hi - lo], non_blocking=True)
                events[b] = torch.cuda.Event()
                events[b].record(stream)
    torch.cuda.current_stream(device).wait_stream(stream)
    return out

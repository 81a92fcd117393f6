"""Tree basis identification for optimal transport (TNET), reference `network_methods/tree_BI.py`.

  max_weight_spanning_tree  -> device: stable radix argsort of the weights, Kruskal order,
                               chunked Kruskal with a lock-free union-find (sx_kruskal); scores of a
                               row-sharded flow (`ShardedScores`): the head of the Kruskal order selected
                               across the shards (sx_order_head_sharded_h), Kruskal on the first shard's GPU
  tree_potentials           -> device: Euler tour + list ranking (sx_tree_potentials); new, the
                               reference reads duals from the LP solver instead
  push_tree_to_bfs          -> device: the tree primal flows (`B x = b[:-1]`, tree_BI.py:74-76, SuperLU in
                               the reference) are subtree sums of b on the same Euler tour
                               (sx_tree_flows, double-double prefix sums);
                               host (native, sx_push_tree_h): the sequential push loop (tree_BI.py:81-110)
                               walks the O(N + pushes) non-zeros instead of a dense S x D scratch.
"""
from __future__ import annotations

import ctypes
from typing import Tuple

import numpy as np

from smart_crossover.formats import OptTransport
from smart_crossover.network_methods.net_manager import (NAN_WEIGHTS_MSG, OTManager, ShardedScores, _SortedFlows,
                                                         _cuda, _dev)
from smart_crossover.output import Basis


def tree_basis_identify(ot_manager: OTManager, flow_weights: np.ndarray) -> Tuple[Basis, int]:
    """Max-weight spanning tree of the flow weights, pushed to a basic feasible solution.
    Returns the basis (last node's row is the redundant one: cbasis = [-1]*(m-1) + [0]) and the
    number of push iterations.  Reference `tree_BI.py:12-29`."""
    # The FULL spanning tree goes to the push phase.  `max_weight_spanning_tree` (like the reference,
    # tree_BI.py:56) drops tree arcs whose weight is exactly zero, after which the reference's square solve
    # (:74-76) fails; the device already has the complete tree, and a zero-weight tree arc is a legitimate
    # (degenerate) basic arc.  Identical to the reference whenever the reference succeeds.
    tree_t, nt = _device_tree(ot_manager.ot, flow_weights, ot_manager._sorted)
    tree = tree_t[:nt].cpu().numpy()
    vbasis, push_iter = push_tree_to_bfs(ot_manager, tree)
    cbasis = np.concatenate([-np.ones(ot_manager.m - 1), np.array([0])])
    return Basis(vbasis, cbasis), push_iter


PREFIX_FACTOR = 16      # the Kruskal order's head handed to the union-find first: 16 N arcs
PREFIX_MIN_ARCS = 1 << 21   # below ~2 M arcs a full argsort is as fast as the prefix path's fixed cost (784^2: 0.25 vs 0.35 ms)


def use_prefix_path(n: int, N: int) -> bool:
    """Whether bare weights go through `sx_kruskal_prefix` (large, dense) or a full argsort."""
    return n >= PREFIX_MIN_ARCS and n > 4 * PREFIX_FACTOR * N


def _device_tree(ot: OptTransport, flow_weights: np.ndarray, _sorted: _SortedFlows = None):
    """(tree arc ids on the device, their number) for the complete bipartite graph of `ot`.

    Large instances first try the head of the Kruskal order only (`sx_kruskal_prefix`: the 16 N
    heaviest arcs, one or two streaming passes instead of a full argsort); the spanning tree is almost
    always complete inside it (SURVEY.md section 6: last tree arc at rank ~8 N).  When the full sort
    already exists (`get_sorted_flows` ran on these weights) the same head is cut from it
    (`sx_kruskal_order_head`).  If the forest is incomplete the whole order is used.  All give the same
    tree: a prefix of a strict total order is unique."""
    dev = _dev()
    S, D = np.shape(ot.M)                 # (.shape of the matrix object: a device-resident one has no host copy)
    N, n = S + D, S * D
    if isinstance(flow_weights, ShardedScores):
        return _sharded_tree(flow_weights, S, D)
    flow_weights = np.asarray(flow_weights, dtype=np.float64)
    have_sort = isinstance(_sorted, _SortedFlows) and _sorted.matches(flow_weights)
    nan_msg = NAN_WEIGHTS_MSG
    if have_sort:
        # NaN keys sort last (NumPy order): one device read instead of an O(n) host scan
        if bool(_sorted.sorted_key[-1:].isnan().item()):
            raise ValueError(nan_msg)
    if not have_sort and use_prefix_path(n, N):
        w_t = _cuda(flow_weights.ravel())
        if bool(w_t.isnan().any().item()):
            raise ValueError(nan_msg)
        head = dev.kruskal_prefix(w_t, PREFIX_FACTOR * N)
        if head is not None:
            tree_t, n_t = dev.kruskal(head, N, S=S, D=D)
            if int(n_t.item()) == N - 1:
                return tree_t, N - 1
        _sorted = _SortedFlows(w_t, flow_weights)
    elif not have_sort:
        _sorted = _SortedFlows(_cuda(flow_weights), flow_weights)
        if bool(_sorted.sorted_key[-1:].isnan().item()):
            raise ValueError(nan_msg)
    if n >= PREFIX_MIN_ARCS and n > 4 * PREFIX_FACTOR * N:
        # the sort exists: only its heaviest 16 N arcs are put into Kruskal order first (one host round trip for
        # the start of the tie run; below ~2 M arcs flipping everything costs less than that round trip)
        head = _sorted.kruskal_order_head(PREFIX_FACTOR * N)
        if head is not None:
            tree_t, n_t = dev.kruskal(head, N, S=S, D=D)
            if int(n_t.item()) == N - 1:
                return tree_t, N - 1
    tree_t, n_t = dev.kruskal(_sorted.kruskal_order(), N, S=S, D=D)
    return tree_t, int(n_t.item())


def _sharded_tree(scores: ShardedScores, S: int, D: int):
    """`_device_tree` for scores held as row shards on several GPUs: the head of the Kruskal order (16 N arcs) is
    selected across the shards and Kruskal runs on the first shard's GPU.  An incomplete forest, or tie runs too
    long for the head's capacity, repeat with 4 x the head until the whole order has been seen."""
    import torch
    dev = _dev()
    N, n = S + D, S * D
    T = PREFIX_FACTOR * N
    with torch.cuda.device(scores.slabs.devices[0]):
        while True:
            head = scores.head(T, kruskal=True)
            tree_t, n_t = dev.kruskal(head, N, S=S, D=D)
            nt = int(n_t.item())
            if nt == N - 1 or head.numel() >= n:
                return tree_t, nt
            T = min(n, 4 * T)


def max_weight_spanning_tree(ot: OptTransport, flow_weights: np.ndarray, _sorted: _SortedFlows = None) -> np.ndarray:
    """Arc ids (ascending) of the maximum-weight spanning tree of K_{S,D}: Kruskal in the order
    'descending weight, ties by ascending arc id'.  Like the reference, tree arcs whose weight is
    exactly zero are dropped from the result (`np.flatnonzero` on the dense tree, tree_BI.py:56)."""
    tree_t, nt = _device_tree(ot, flow_weights, _sorted)
    tree = tree_t[:nt].cpu().numpy()
    w = flow_weights.take(tree) if isinstance(flow_weights, ShardedScores) else np.asarray(flow_weights)[tree]
    return tree[w != 0]


def tree_potentials(ot: OptTransport, tree: np.ndarray) -> np.ndarray:
    """Duals y of the tree basis: y[S+j] - y[i] = M[i, j] on tree arcs, y[last node] = 0
    (B^T y[:-1] = c[tree]; reference gets these from the solver, algorithms.py:132)."""
    dev = _dev()
    M = np.asarray(ot.M, dtype=np.float64)
    S, D = M.shape
    y = dev.tree_potentials(_cuda(np.asarray(tree, dtype=np.int64)), int(len(tree)), S + D, _cuda(M), S + D - 1, S=S, D=D)
    return y.cpu().numpy()


def tree_flows(ot: OptTransport, tree: np.ndarray) -> np.ndarray:
    """Primal flows of the tree basis, one per tree arc: B x = b[:-1] with B = A[:-1, tree] and
    b = [-s, d] (reference tree_BI.py:74-76).  Needs a spanning tree (N - 1 arcs)."""
    dev = _dev()
    S, D = ot.s.size, ot.d.size
    tree = np.asarray(tree, dtype=np.int64)
    b = np.hstack([-np.asarray(ot.s, dtype=np.float64), np.asarray(ot.d, dtype=np.float64)])
    return dev.tree_flows(_cuda(tree), int(tree.size), S + D, _cuda(b), S + D - 1, S=S, D=D).cpu().numpy()


def push_tree_to_bfs(ot_manager: OTManager, tree: np.ndarray, _flows: np.ndarray = None) -> Tuple[np.ndarray, int]:
    """Tree primal flows, then 'irrigation' pushes until no tree flow is negative.
    Returns (vbasis, push_iter) with vbasis = 0 on arcs carrying positive flow, -1 elsewhere.
    `_flows` (tests of the host loop) supplies the tree flows instead of computing them on the GPU."""
    ot = ot_manager.ot
    S, D = ot.s.size, ot.d.size
    tree = np.asarray(tree, dtype=np.int64)
    flow = np.asarray(_flows, dtype=np.float64) if _flows is not None else tree_flows(ot, tree)

    # the push loop itself is sequential host work on the sparse support (libsxcross, sx_push_tree_h)
    from smart_crossover import _native
    tree = np.ascontiguousarray(tree, dtype=np.int64)
    flow = np.ascontiguousarray(flow, dtype=np.float64)
    cap = 2 * int(tree.size) + 1024
    while True:
        pos = np.empty(cap, dtype=np.int64)
        n_pos, push_iter = ctypes.c_int64(0), ctypes.c_int64(0)
        rc = _native.lib.sx_push_tree_h(tree.ctypes.data, flow.ctypes.data, int(tree.size), S, D, pos.ctypes.data, cap,
                                        ctypes.byref(n_pos), ctypes.byref(push_iter))
        if rc == _native.SX_ERR_WORKSPACE:                       # more corners were created than guessed
            cap = int(n_pos.value)
            continue
        if rc == _native.SX_ERR_PUSH_ASSERT:                     # the reference asserts here (tree_BI.py:93-94)
            raise AssertionError("push_tree_to_bfs: no positive flow to push against (reference tree_BI.py:93-94)")
        _native.check(rc, "sx_push_tree_h")
        break
    vbasis = -np.ones(ot_manager.n)
    vbasis[pos[:n_pos.value]] = 0
    return vbasis, int(push_iter.value)

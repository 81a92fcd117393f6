"""First-order warm start for the OT crossover: an entropic Sinkhorn point computed on the GPU.

The reference's experiment driver calls POT for it, `ot.sinkhorn(ot.s, ot.d, ot.M, reg=10,
numItermax=1000)` (`scripts/run_network_crossover.py:96`), and hands the flattened plan to
`network_crossover`.  POT is not part of the reference tree; `sinkhorn` below keeps its call shape
(marginals, cost matrix, `reg`, `numItermax`, `stopThr`; returns the S x D plan) and runs the same
Sinkhorn-Knopp iteration in the log domain on the device (`sx_sinkhorn_ot`, csrc/sx_sinkhorn.cu).
A cost matrix held as `device.CostSlabs` (row shards on several GPUs, e.g. the slabs of
`OTManager.from_device_cost`) runs the same iteration on every shard's GPU (`sx_sinkhorn_ot_sharded_h`).
"""
from __future__ import annotations

import ctypes

import numpy as np


def sinkhorn(a, b, M, reg: float, numItermax: int = 1000, stopThr: float = 1e-9, log: bool = False,
             as_slabs: bool = False):
    """Entropic-regularised OT plan gamma = diag(u) exp(-M / reg) diag(v) between marginals a (S,)
    and b (D,).  With log=True also returns {'niter', 'err', 'f', 'g'} (potentials reg*log u, reg*log v).
    as_slabs (M a `device.CostSlabs` only): return the plan as row slabs on M's devices (`CostSlabs` with
    contiguous rows, the flow `OTManager.get_sorted_flows` scores shard by shard) instead of a host array."""
    import torch
    from smart_crossover import device as dev
    from smart_crossover._native import check, lib

    dev._require_cuda()
    if isinstance(M, dev.CostSlabs):
        return _sinkhorn_slabs(a, b, M, reg, numItermax, stopThr, log, as_slabs)
    if as_slabs:
        raise ValueError("as_slabs needs the cost matrix as device.CostSlabs")
    a_t, b_t = dev._f64(np.asarray(a, dtype=np.float64)), dev._f64(np.asarray(b, dtype=np.float64))
    M_t = dev._f64(M) if not (isinstance(M, torch.Tensor) and M.is_cuda) else M.contiguous()
    S, D = M_t.shape
    if a_t.numel() != S or b_t.numel() != D:
        raise ValueError("marginals do not match the cost matrix")
    f = torch.empty(S, dtype=torch.float64, device=M_t.device)
    g = torch.empty(D, dtype=torch.float64, device=M_t.device)
    X = torch.empty(S, D, dtype=torch.float64, device=M_t.device)
    ws = dev._ws(lib.sx_sinkhorn_workspace_bytes(S, D), M_t.device)
    iters, err = ctypes.c_int64(0), ctypes.c_double(0.0)
    check(lib.sx_sinkhorn_ot(dev._ptr(M_t), M_t.stride(0), S, D, dev._ptr(a_t), dev._ptr(b_t), float(reg),
                             int(numItermax), float(stopThr), 10, dev._ptr(f), dev._ptr(g), dev._ptr(X),
                             ctypes.byref(iters), ctypes.byref(err), dev._ptr(ws), ws.numel(), dev._stream()),
          "sx_sinkhorn_ot")
    plan = X.cpu().numpy()
    if log:
        return plan, {"niter": iters.value, "err": err.value, "f": f.cpu().numpy(), "g": g.cpu().numpy()}
    return plan


def _sinkhorn_slabs(a, b, slabs, reg, numItermax, stopThr, log, as_slabs):
    """`sinkhorn` over the row shards of a `device.CostSlabs`: shard g's rows on its device, the plan assembled on
    the host shard by shard (or left in place with as_slabs).  The cost matrix is never read on the host."""
    from smart_crossover import device as dev
    from smart_crossover._native import check, lib

    S, D, G = slabs.S, slabs.D, len(slabs.devices)
    a = np.ascontiguousarray(a, dtype=np.float64).ravel()
    b = np.ascontiguousarray(b, dtype=np.float64).ravel()
    if a.size != S or b.size != D:
        raise ValueError("marginals do not match the cost matrix")
    X = dev.CostSlabs(S, D, slabs.devices, slabs.row_bounds, pad_ld=False)
    f, g_pot = np.empty(S), np.empty(D)
    slabs.sync()
    iters, err = ctypes.c_int64(0), ctypes.c_double(0.0)
    check(lib.sx_sinkhorn_ot_sharded_h(G, (ctypes.c_int * G)(*slabs.devices),
                                       (ctypes.c_void_p * G)(*[t.data_ptr() for t in slabs.t]),
                                       (ctypes.c_int64 * (G + 1))(*slabs.row_bounds), slabs.ld, S, D,
                                       a.ctypes.data, b.ctypes.data, float(reg), int(numItermax), float(stopThr), 10,
                                       f.ctypes.data, g_pot.ctypes.data,
                                       (ctypes.c_void_p * G)(*[x.data_ptr() for x in X.t]),
                                       ctypes.byref(iters), ctypes.byref(err)), "sx_sinkhorn_ot_sharded_h")
    if as_slabs:
        plan = X
    else:
        plan = np.empty((S, D))
        for g in range(G):
            plan[slabs.row0[g]:slabs.row0[g] + slabs.rows[g]] = dev.to_host(X.t[g])
    if log:
        return plan, {"niter": iters.value, "err": err.value, "f": f, "g": g_pot}
    return plan

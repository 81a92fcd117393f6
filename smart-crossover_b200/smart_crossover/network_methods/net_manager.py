"""Problem managers of the network crossover: `OTManager`, `MCFManagerStd`, `NetworkManager`.

Same public surface as the reference (`network_methods/net_manager.py:14-509`): the nine
protocol methods plus the concrete extras the driver uses (`get_mcf`, `extend_by_bigM`,
`set_initial_basis`, `rescale_cost`, `fix_variables`, `get_reduced_cost_for_original_OT/_mcf`,
`get_sub_problem`, `get_X`) and the public fields (`ot`, `mcf`, `mask_sub_ot`,
`artificial_vars`, `var_info`, `c_rescaling_factor`).  What changed is where the arithmetic
runs:

  get_sorted_flows                      -> sx_score_ot / sx_score_mcf + sx_argsort_f64 (device)
  get_reduced_cost_for_original_* and
  check_optimality_condition            -> sx_price_dense_ot / sx_price_arcs (device), fused count
  price (new; north_star top-k)         -> + sx_topk_select

The problem data (cost matrix or arc list) is uploaded to the GPU once, on first use, and stays
resident; per call only the duals go up and a few hundred bytes come back.  Sub-problem
extraction, basis bookkeeping and the LP re-solve stay on the host, as in the reference; the
restricted master is assembled directly from arc ids instead of slicing the full 2n-nonzero
incidence matrix every round (`net_manager.py:450-455`).  There is no CPU fallback for the
device steps: without a CUDA device they raise.
"""
from __future__ import annotations

from typing import Tuple

import numpy as np
import scipy.sparse as sp
from typing_extensions import Protocol

from smart_crossover.formats import MinCostFlow, OptTransport
from smart_crossover.output import Basis, Output
from smart_crossover.parameters import TOLERANCE_FOR_ARTIFICIAL_VARS, TOLERANCE_FOR_REDUCED_COSTS
from smart_crossover.solver_caller.caller import SolverSettings
from smart_crossover.solver_caller.solving import solve_mcf


class NetworkManager(Protocol):
    """What `column_generation` needs from a manager (reference `net_manager.py:14-113`)."""

    m: int
    n: int
    basis: Basis

    def get_sorted_flows(self, x: np.ndarray) -> Tuple[np.ndarray, np.ndarray]: ...
    def recover_x_from_sub_x(self, x_sub: np.ndarray) -> np.ndarray: ...
    def recover_basis_from_sub_basis(self, basis_sub: Basis) -> Basis: ...
    def solve_subproblem(self, solver: str, solver_settings: SolverSettings) -> Output: ...
    def recover_obj_val(self, obj_val: float) -> float: ...
    def check_optimality_condition(self, x: np.ndarray, y: np.ndarray) -> bool: ...
    def add_free_variables(self, ind_free: np.ndarray) -> None: ...
    def update_subproblem(self) -> None: ...
    def set_basis(self, basis: Basis) -> None: ...


def _dev():
    """The device operators; importing them needs torch + libsxcross and fails loudly otherwise."""
    from smart_crossover import device
    return device


def _cuda(a, dtype=None):
    """Host array -> tensor on the current device (large arrays through pinned staging, `device.to_device`)."""
    return _dev().to_device(np.asarray(a), dtype=dtype)


class BigMExtendedCost:
    """(S+1) x (D+1) cost matrix of the big-M extension (reference `net_manager.py:390-393`: last column and
    last row = bigM, corner = 0) as a VIEW of the original matrix: nothing is copied until somebody asks for
    the dense array (`np.asarray`), which the managers never do -- the sub-problem takes single entries
    (`take_flat`) and the device builds its own extended copy (`CostSlabs.from_host(border=...)`).

    The base may be a `DeviceResidentCost`: `take_flat` then gathers inner entries from its slabs, the device
    prices the extension over those slabs (`device.OTPricer(..., bigm=)`), and there is no dense array."""

    ndim = 2
    dtype = np.dtype(np.float64)

    def __init__(self, base, bigM: float) -> None:
        self.base = base if isinstance(base, DeviceResidentCost) else np.asarray(base)
        self.bigM = float(bigM)
        self.shape = (self.base.shape[0] + 1, self.base.shape[1] + 1)
        self.size = self.shape[0] * self.shape[1]

    def take_flat(self, ids: np.ndarray) -> np.ndarray:
        """Entries at row-major indices `ids` of the extended matrix."""
        S, D = self.base.shape
        i, j = np.divmod(np.asarray(ids, dtype=np.int64), D + 1)
        inner = (i < S) & (j < D)
        out = np.full(i.shape, self.bigM)
        if isinstance(self.base, DeviceResidentCost):
            out[inner] = self.base.take_flat(i[inner] * D + j[inner])
        else:
            out[inner] = self.base[i[inner], j[inner]]
        out[(i == S) & (j == D)] = 0.0
        return out

    def __array__(self, dtype=None, copy=None):
        if isinstance(self.base, DeviceResidentCost):
            return np.asarray(self.base)                # raises: a device-resident base has no host copy
        S, D = self.base.shape
        M = np.full(self.shape, self.bigM)
        M[:S, :D] = self.base
        M[S, D] = 0.0
        return M if dtype is None else M.astype(dtype, copy=False)

    def __getitem__(self, key):
        if isinstance(key, tuple) and len(key) == 2 and all(isinstance(k, (int, np.integer)) for k in key):
            i, j = (int(k) % n for k, n in zip(key, self.shape))
            return float(self.take_flat(np.array([i * self.shape[1] + j]))[0])
        return np.asarray(self)[key]

    def ravel(self):
        return np.asarray(self).ravel()

    flatten = ravel

    def max(self, axis=None, out=None):
        if axis is not None or out is not None:
            raise ValueError("only the maximum over all entries is available")
        return max(float(self.base.max()), self.bigM, 0.0)


class DeviceResidentCost:
    """Stand-in for `ot.M` when the cost matrix only exists on the device(s) (`OTManager.from_device_cost`:
    a 60 000 x 60 000 matrix generated shard by shard in HBM has no host copy).  Knows its shape; any attempt
    to read it on the host raises."""

    ndim = 2
    dtype = np.dtype(np.float64)

    def __init__(self, slabs) -> None:
        self.slabs = slabs
        self.shape = (slabs.S, slabs.D)
        self.size = slabs.S * slabs.D

    def take_flat(self, ids: np.ndarray) -> np.ndarray:
        """Entries at row-major arc ids, gathered from the device shards (the restricted master's costs)."""
        return self.slabs.take_flat(ids)

    def max(self, axis=None, out=None):
        """Largest entry, taken on the shards' devices (what `np.max(cost)` calls); NaN if any entry is NaN."""
        if axis is not None or out is not None:
            raise ValueError("a device-resident cost matrix only gives its maximum over all entries")
        return self.slabs.max()

    def __array__(self, dtype=None, copy=None):
        raise TypeError("this cost matrix is device resident; it has no host copy")


def _take_flat(M, ids: np.ndarray) -> np.ndarray:
    if isinstance(M, DeviceResidentCost):
        return M.take_flat(ids)
    return M.take_flat(ids) if isinstance(M, BigMExtendedCost) else np.asarray(M).ravel()[ids]


class _SortedFlows:
    """Device-resident result of one `get_sorted_flows` call, kept so that the tree build
    (`tree_BI.max_weight_spanning_tree`) can reuse the sort instead of repeating it.
    `scores_np = None`: the scores are downloaded here, on a copy stream, WHILE the sort runs."""

    def __init__(self, scores_t, scores_np=None):
        import torch
        dev = _dev()
        self.scores_t = scores_t
        ready = torch.cuda.Event()
        ready.record()                                   # the scores are complete; the sort is enqueued after this
        self.order, self.sorted_key = dev.argsort_f64(scores_t)
        self.scores_np = scores_np if scores_np is not None else dev.to_host(scores_t, ready=ready)

    def queue(self) -> np.ndarray:
        dev = _dev()
        return dev.to_host(dev.queue_from_order(self.order))

    def kruskal_order(self):
        return _dev().kruskal_order(self.sorted_key, self.order)

    def kruskal_order_head(self, T: int):
        """The first >= T arcs of the Kruskal order (whole tie runs), or None if the runs are too long."""
        return _dev().kruskal_order_head(self.sorted_key, self.order, T)

    def matches(self, weights: np.ndarray) -> bool:
        """Whether `weights` are the scores this sort was made from: the very array `get_sorted_flows`
        returned, or a view of it.  (No O(n) host comparison: at 3.6e9 arcs that would cost more than the
        tree build; a caller that passes a modified copy simply gets a fresh sort.)"""
        return weights is self.scores_np or (isinstance(weights, np.ndarray) and weights.size == self.scores_np.size
                                             and np.shares_memory(weights, self.scores_np))


NAN_WEIGHTS_MSG = "flow weights contain NaN (a zero marginal?): the spanning tree is undefined"


class ShardedScores:
    """Flow indicators of a row-sharded flow, left on the devices that hold its shards: the sharded counterpart of
    `_SortedFlows`, and what `OTManager.get_sorted_flows` returns as the scores of a flow given as slabs.  Nothing
    sorts all n arcs: `head` selects the first arcs of either order across the shards (`sx_order_head_sharded_h`).
    A handle, not an array: `shape`, `len`, `take(ids)`; converting it to a host array raises."""

    ndim = 1
    dtype = np.dtype(np.float64)

    def __init__(self, slabs, hists=None) -> None:
        self.slabs, self.hists = slabs, hists
        self.size = slabs.S * slabs.D
        self.shape = (self.size,)
        self._nan = None

    def __len__(self) -> int:
        return self.size

    def __array__(self, dtype=None, copy=None):
        raise TypeError("these flow scores are device resident; they have no host copy")

    def take(self, ids: np.ndarray) -> np.ndarray:
        """Scores of the arcs `ids` (host float64)."""
        return self.slabs.take_flat(ids)

    def has_nan(self) -> bool:
        """Whether any score is NaN.  NaN and +inf share the top bin of the level-0 histograms, so only shards with
        something there are scanned."""
        if self._nan is None:
            nan = False
            for g, t in enumerate(self.slabs.t):
                if self.hists is None or int(self.hists[g][4095].item()) != 0:
                    nan = nan or bool(t.isnan().any().item())
            self._nan = nan
        return self._nan

    def head(self, T: int, kruskal: bool, T_cap: int | None = None):
        """At least min(T, n) arcs at the head of the Kruskal order (kruskal=True: uint32 ids as int32) or of the
        queue (int64), on the first shard's device.  When the tie runs at the threshold do not fit T_cap the call
        is repeated with 4 x T_cap; beyond the first device's memory it raises MemoryError."""
        from smart_crossover import device as dev
        from smart_crossover._native import SxError, lib
        import torch
        if self.has_nan():
            raise ValueError(NAN_WEIGHTS_MSG)
        n = self.size
        T = int(min(T, n))
        T_cap = int(min(n, T_cap or max(2 * T, T + 65536)))
        while True:
            try:
                out = dev.order_head_sharded(self.slabs, T, T_cap, self.hists, queue=not kruskal)
            except (torch.OutOfMemoryError, SxError) as e:
                if isinstance(e, SxError) and not (e.code == -2 and lib.sx_last_cuda_error() == 2):
                    raise
                raise MemoryError(f"the head of {T} arcs (capacity {T_cap}) of the flow order does not fit on "
                                  f"device {self.slabs.devices[0]}") from e
            if out is not None:
                return out
            T_cap = min(n, 4 * T_cap)


class ShardedQueue:
    """The arcs of a sharded flow sorted by score, largest first (ties by descending arc id), as `column_generation`
    reads it: `len(queue) == n` and `queue[a:b]` is the int64 host array the host path's queue gives.  Only the
    head that slices have reached is materialised (`ShardedScores.head` in queue mode), grown geometrically."""

    def __init__(self, scores: ShardedScores) -> None:
        self.scores = scores
        self._head = np.empty(0, dtype=np.int64)

    def __len__(self) -> int:
        return self.scores.size

    def __getitem__(self, key) -> np.ndarray:
        if not isinstance(key, slice):
            raise TypeError("a sharded queue is read in slices")
        a, b, step = key.indices(len(self))
        if step != 1:
            raise ValueError("a sharded queue is read in slices of step 1")
        if b > self._head.size:
            T = min(len(self), max(b, 2 * self._head.size, 1 << 16))
            self._head = self.scores.head(T, kruskal=False).cpu().numpy()
        return self._head[a:max(a, b)].copy()


# =================================================================================================
class OTManager:
    """Optimal-transport manager (reference `net_manager.py:322-509`).

    After `extend_by_bigM` the host-side `ot` is the (S+1) x (D+1) extended problem as in the reference,
    but its cost matrix is a view (`BigMExtendedCost`), not a copy; the device builds the extended matrix
    itself from the original block, so the S + D + 1 artificial arcs are priced by the same kernel as
    everything else and arc ids come back in the extended numbering.  A device-resident matrix keeps its slabs
    and the pricer prices the border next to them (`device.OTPricer(..., bigm=)`), with the same ids and results.
    """

    def __init__(self, ot: OptTransport) -> None:
        self.ot = ot
        self.m = ot.s.size + ot.d.size
        self.n = ot.s.size * ot.d.size
        self.mask_sub_ot = np.zeros(self.n, dtype=bool)
        self.artificial_vars = np.array([])
        self._slabs = None              # device-resident row shards of the CURRENT cost matrix (built on first pricing)
        self._pricers = {}              # K -> persistent OTPricer over those shards
        self._mcf = None
        self._sorted = None
        self._bigM = None
        if isinstance(ot.M, DeviceResidentCost):
            self._slabs = ot.M.slabs
        elif isinstance(ot.M, BigMExtendedCost) and isinstance(ot.M.base, DeviceResidentCost):
            self._slabs, self._bigM = ot.M.base.slabs, ot.M.bigM

    @classmethod
    def from_device_cost(cls, s: np.ndarray, d: np.ndarray, slabs) -> "OTManager":
        """Manager over a cost matrix that already sits on the device(s) as `device.CostSlabs` (generated or
        uploaded there by the caller).  Scoring, the tree build, pricing and the restricted master work as
        usual.  `extend_by_bigM` keeps the slabs: the border of the extension is priced on the devices next to
        them (`device.OTPricer(..., bigm=)`), so `cnet_ot` runs without a second, extended copy of the matrix.
        `to_MCF` / `get_mcf` need the host matrix and are not available."""
        return cls(OptTransport(np.asarray(s, dtype=np.float64), np.asarray(d, dtype=np.float64),
                                DeviceResidentCost(slabs)))

    # ---- lazily built host / device state ---------------------------------------------------------
    @property
    def mcf(self) -> MinCostFlow:
        """MCF form of the current OT (`get_mcf`, reference :353-355); built on first access."""
        if self._mcf is None:
            self._mcf = self.ot.to_MCF()
        return self._mcf

    @mcf.setter
    def mcf(self, value) -> None:
        self._mcf = value

    def get_mcf(self) -> None:
        self._mcf = self.ot.to_MCF()

    def _device_slabs(self):
        """The cost matrix on the device(s), uploaded once per problem: row-sharded over the GPUs
        `device.pricing_devices` picks (one below ~3e7 arcs per extra GPU).  After `extend_by_bigM` the
        device matrix is the extended one, built on the device from the original block."""
        if self._slabs is None:
            dev = _dev()
            S, D = self.ot.s.size, self.ot.d.size
            devices = dev.pricing_devices(S * D, S)
            if isinstance(self.ot.M, BigMExtendedCost):
                self._slabs = dev.CostSlabs.from_host(self.ot.M.base, devices, border=(self.ot.M.bigM, 0.0))
            else:
                self._slabs = dev.CostSlabs.from_host(self.ot.M, devices)
        return self._slabs

    def _border(self):
        """(bigM, corner) when the device slabs are the base of the big-M extension (a device-resident problem after
        `extend_by_bigM`), else None."""
        M = self.ot.M
        if isinstance(M, BigMExtendedCost) and isinstance(M.base, DeviceResidentCost):
            return M.bigM, 0.0
        return None

    def _pricer(self, K: int):
        """One persistent pricer per top-K size (buffers, streams and worker threads live as long as the
        manager: a column-generation round allocates nothing)."""
        pr = self._pricers.get(K)
        if pr is None:
            pr = self._pricers[K] = _dev().OTPricer(self._device_slabs(), K, tol=TOLERANCE_FOR_REDUCED_COSTS,
                                                    bigm=self._border())
        return pr

    def _drop_device_state(self, keep_slabs: bool = False):
        for pr in self._pricers.values():
            pr.close()
        self._pricers = {}
        if not keep_slabs:
            self._slabs = None

    def pricing_devices(self):
        """Devices the cost matrix is sharded over (diagnostics)."""
        return list(self._device_slabs().devices)

    def get_X(self, x: np.ndarray) -> np.ndarray:
        return x.reshape((self.ot.s.size, self.ot.d.size))

    # ---- K1: scores + sorted queue --------------------------------------------------------------------
    def get_sorted_flows(self, x: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
        """Flow indicators max(x_ij/s_i, x_ij/d_j) and the arcs sorted by them, largest first
        (stable sort: ties by descending arc id).  Reference :368-379.

        `x` may also be the flow as row slabs (`device.CostSlabs`, e.g. `warm_start.sinkhorn(..., as_slabs=True)`)
        with the devices and row bounds of the manager's cost slabs.  Each shard is then scored on its own GPU and
        the call returns a lazy `ShardedQueue` and the device-resident `ShardedScores`: no n-sized array is sorted
        or crosses PCIe."""
        dev = _dev()
        if isinstance(x, dev.CostSlabs):
            # (compared with the slabs already on the devices: a host cost matrix is not uploaded just to refuse x)
            if self._slabs is None or not x.same_shards(self._slabs):
                raise ValueError("the flow slabs must have the cost slabs' shape, devices and row bounds")
            self._sorted = ShardedScores(*dev.score_ot_slabs(x, self.ot.s, self.ot.d))
            return ShardedQueue(self._sorted), self._sorted
        scores_t = dev.score_ot(_cuda(np.asarray(x, dtype=np.float64).ravel()),
                                _cuda(np.asarray(self.ot.s, dtype=np.float64)),
                                _cuda(np.asarray(self.ot.d, dtype=np.float64)))
        self._sorted = _SortedFlows(scores_t)
        return self._sorted.queue(), self._sorted.scores_np

    # ---- big-M extension ----------------------------------------------------------------------------------
    def extend_by_bigM(self, bigM: float) -> None:
        """Artificial source and sink joined to everything at cost bigM (reference :381-400)."""
        S, D = self.ot.s.size, self.ot.d.size
        mask = np.zeros((S + 1, D + 1), dtype=np.bool_)
        mask[S, :] = True
        mask[:, D] = True
        self.mask_sub_ot = mask
        # row-major ids of the border, ascending (= np.where(mask.ravel())[0] without scanning n booleans)
        self.artificial_vars = np.concatenate([np.arange(S, dtype=np.int64) * (D + 1) + D,
                                               S * (D + 1) + np.arange(D + 1, dtype=np.int64)])
        self._bigM = float(bigM)
        # `ot.M` becomes a view of the extended matrix: neither the host nor the PCIe link ever sees a copy.  A
        # device-resident matrix keeps its slabs; the pricers built next price the border next to them.
        device_resident = isinstance(self.ot.M, DeviceResidentCost)
        self.ot = OptTransport(np.append(self.ot.s, np.sum(self.ot.d)),
                               np.append(self.ot.d, np.sum(self.ot.s)), BigMExtendedCost(self.ot.M, bigM))
        self._drop_device_state(keep_slabs=device_resident)
        self._mcf = None
        self._sorted = None

    # ---- sub-problem bookkeeping (host) ---------------------------------------------------------------------
    def add_free_variables(self, ind_free: np.ndarray) -> None:
        """Open columns of the restricted master.  Accepts arc ids of the ORIGINAL problem or, as the
        `tnet` driver passes (algorithms.py:58), a boolean mask over them.  Reference :402-414."""
        if self.artificial_vars.size > 0:
            inner = self.mask_sub_ot[:-1, :-1]
            rows, cols = np.unravel_index(ind_free, inner.shape)
            inner[rows, cols] = True
        else:
            self.mask_sub_ot[np.asarray(ind_free).ravel()] = True

    def set_basis(self, basis: Basis) -> None:
        self.basis = basis

    def recover_x_from_sub_x(self, x_sub: np.ndarray) -> np.ndarray:
        x = np.zeros(self.ot.s.size * self.ot.d.size)
        x[self.mask_sub_ot.ravel()] = x_sub
        return x

    def recover_basis_from_sub_basis(self, basis_sub: Basis) -> Basis:
        vbasis = -np.ones(self.ot.s.size * self.ot.d.size)
        vbasis[self.mask_sub_ot.ravel()] = basis_sub.vbasis
        return Basis(vbasis, basis_sub.cbasis)

    def get_sub_problem(self) -> MinCostFlow:
        """Restricted master over the open columns (ascending arc id), assembled straight from the
        arc ids: column k = (i, j) has -1 at row i and +1 at row S + j.  Equals the reference's
        `self.mcf.A.tocsc()[:, mask]` (:450-455) without touching the full matrix."""
        S, D = self.ot.s.size, self.ot.d.size
        ids = np.flatnonzero(self.mask_sub_ot.ravel())
        k = ids.size
        rows = np.empty(2 * k, dtype=np.int64)
        rows[0::2] = ids // D
        rows[1::2] = S + ids % D
        vals = np.empty(2 * k)
        vals[0::2] = -1.0
        vals[1::2] = 1.0
        A = sp.csc_matrix((vals, rows, np.arange(0, 2 * k + 1, 2)), shape=(S + D, k))
        return MinCostFlow(A=A, b=np.hstack([-self.ot.s, self.ot.d]),
                           c=_take_flat(self.ot.M, ids), u=np.full(k, np.inf))

    def solve_subproblem(self, solver: str, solver_settings: SolverSettings) -> Output:
        method = "network_simplex" if solver == "CPL" else "default"
        warm = Basis(self.basis.vbasis[self.mask_sub_ot.ravel()], self.basis.cbasis)
        return solve_mcf(self.get_sub_problem(), solver=solver, method=method, warm_start_basis=warm,
                         settings=solver_settings)

    def recover_obj_val(self, obj_val):
        return obj_val

    def update_subproblem(self):
        """Nothing to rebuild for OT: the open columns live in `mask_sub_ot` (reference :499-501)."""

    def set_initial_basis(self) -> None:
        vbasis = -np.ones(self.ot.s.size * self.ot.d.size)
        vbasis[self.artificial_vars] = 0
        self.basis = Basis(vbasis, np.concatenate([-np.ones(self.m + 1), np.zeros(1)]))

    # ---- K4: pricing ---------------------------------------------------------------------------------------------
    def price(self, y: np.ndarray, K: int = 0, want_rc: bool = False):
        """One pricing pass over every arc of the current OT (after `extend_by_bigM`: the extended one):
        violator count, min reduced cost and the K most violating arcs (north_star extension; see
        `device.PriceResult`).  Goes through the manager's persistent, row-sharded pricer: the duals are the
        only upload.  `want_rc` also returns the full reduced-cost vector (host), shard by shard."""
        y = np.asarray(y, dtype=np.float64)
        S, D = self.ot.s.size, self.ot.d.size
        res = self._pricer(int(K)).price(y[:S], y[S:S + D])
        if want_rc:
            import torch
            dev = _dev()
            slabs = self._device_slabs()
            Sb, Db = slabs.S, slabs.D                  # the slabs' own shape: (S - 1, D - 1) when they are the base
            rc = np.empty((S, D))
            for g, d in enumerate(slabs.devices):
                with torch.cuda.device(d):
                    r0, rows = slabs.row0[g], slabs.rows[g]
                    y_g = torch.from_numpy(np.concatenate([y[r0:r0 + rows], y[S:S + Db]])).cuda()
                    part = dev.price_dense_ot(slabs.view(g), y_g, K=0, tol=TOLERANCE_FOR_REDUCED_COSTS, want_rc=True)
                    rc[r0:r0 + rows, :Db] = part.rc.cpu().numpy().reshape(rows, Db)
            border = self._border()
            if border is not None:
                # the S + D + 1 border arcs, associated as the kernels do: c - (v_j - u_i)
                bigM, corner = border
                u, v = y[:S], y[S:S + D]
                rc[:Sb, Db] = bigM - (v[Db] - u[:Sb])
                rc[Sb, :Db] = bigM - (v[:Db] - u[Sb])
                rc[Sb, Db] = corner - (v[Db] - u[Sb])
            res.rc = rc.ravel()
        return res

    def get_reduced_cost_for_original_OT(self, y: np.ndarray) -> np.ndarray:
        """rc = c - A^T y over every arc of the current OT (reference :474-483)."""
        return self.price(y, K=0, want_rc=True).rc

    def check_optimality_condition(self, x: np.ndarray, y: np.ndarray) -> bool:
        """All reduced costs >= -1e-6 and no flow left on artificial arcs (reference :485-497)."""
        art_ok = bool(np.all(x[self.artificial_vars][:-1] < TOLERANCE_FOR_ARTIFICIAL_VARS)) \
            if self.artificial_vars.size > 0 else True
        return bool(art_ok and self.price(y, K=0).optimal)


# =================================================================================================
class MCFManagerStd:
    """Min-cost-flow manager (reference `net_manager.py:116-319`)."""

    def __init__(self, mcf: MinCostFlow) -> None:
        self.mcf = mcf
        self.m = self.mcf.b.size
        self.n = self.mcf.c.size
        self.var_info = {"non_fix": np.arange(self.n, dtype=np.int64)}
        self.artificial_vars = np.array([])
        self.c_rescaling_factor = None
        self._arcs_dev = None
        self._sorted = None
        self._arc_pricers = {}          # K -> reusable pricing buffers
        self._vb_src, self._vb_dev = None, None
        self._host_arcs_of, self._host_tail, self._host_head = None, None, None
        self._freed = None              # bool over the arcs: opened by add_free_variables so far

    # ---- arc list of the current incidence matrix (host scan once per matrix, then device resident) ------
    @staticmethod
    def _endpoints(A) -> Tuple[np.ndarray, np.ndarray]:
        """tail = row of the +1, head = row of the -1 of every column (`scripts/min2mcf.py:36-37`);
        -1 where a column lacks that entry."""
        A = sp.csc_matrix(A)
        E = A.shape[1]
        cols = np.repeat(np.arange(E, dtype=np.int64), np.diff(A.indptr))
        tail = np.full(E, -1, dtype=np.int64)
        head = np.full(E, -1, dtype=np.int64)
        tail[cols[A.data > 0]] = A.indices[A.data > 0]
        head[cols[A.data < 0]] = A.indices[A.data < 0]
        return tail, head

    def _host_arcs(self) -> Tuple[np.ndarray, np.ndarray]:
        """(tail, head) of every column of the current `mcf.A`: one host scan per matrix (the big-M extension
        appends its arcs without a scan)."""
        if self._host_arcs_of is not self.mcf.A:
            tail, head = self._endpoints(self.mcf.A)
            if (tail < 0).any() or (head < 0).any():
                raise ValueError("every column of A must have one +1 and one -1 entry")
            self._host_arcs_of, self._host_tail, self._host_head = self.mcf.A, tail, head
        return self._host_tail, self._host_head

    def _device_arcs(self):
        import torch
        if self._arcs_dev is None or self._arcs_dev["A"] is not self.mcf.A:
            tail, head = self._host_arcs()
            self._arcs_dev = {"A": self.mcf.A, "tail": _cuda(tail, torch.int32), "head": _cuda(head, torch.int32),
                              "c": None, "c_src": None}
        d = self._arcs_dev
        if d["c_src"] is not self.mcf.c:
            d["c"] = _cuda(np.asarray(self.mcf.c, dtype=np.float64))
            d["c_src"] = self.mcf.c
        return d

    # ---- K1 -----------------------------------------------------------------------------------------------------
    def get_sorted_flows(self, x: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
        """Flow indicators after reversing arcs with x > u/2, and the arcs sorted by them, largest
        first (stable).  Reference :156-184; needs finite capacities (u = inf gives NaN there too)."""
        import torch
        dev = _dev()
        A = self.mcf.A.tocsr()
        if not A.has_sorted_indices:
            A = A.sorted_indices()
        arcs = self._device_arcs()
        scores_t = dev.score_mcf(_cuda(np.asarray(x, dtype=np.float64)), _cuda(np.asarray(self.mcf.u, dtype=np.float64)),
                                 arcs["tail"], arcs["head"], _cuda(A.indptr, torch.int64),
                                 _cuda(A.indices, torch.int32), _cuda(np.sign(A.data), torch.int8))
        self._sorted = _SortedFlows(scores_t)
        return self._sorted.queue(), self._sorted.scores_np

    # ---- big-M extension, rescaling, fixing (host) -----------------------------------------------------------------
    def extend_by_bigM(self, bigM: float) -> None:
        """One artificial node joined to every node by an arc of cost bigM, oriented so that it can
        absorb that node's residual supply once the fixed-at-upper arcs are accounted for
        (reference :135-154)."""
        at_up = np.zeros(self.n, dtype=bool)
        at_up[self.var_info["fix_up"]] = True
        b_true = self.mcf.b - self.mcf.A.multiply(at_up) @ (self.mcf.u * at_up)
        sign = np.sign(b_true)
        sign[sign == 0] = 1
        tail, head = self._host_arcs()
        A_ext = sp.vstack((sp.hstack((self.mcf.A, sp.diags(sign))),
                           sp.csr_matrix(np.concatenate([np.zeros(self.n), -sign]))))
        # the reference sizes the artificial capacities with n instead of m (:148, harmless); m is used here
        self.mcf = MinCostFlow(A_ext, np.append(self.mcf.b, 0.0),
                               np.concatenate([self.mcf.c, bigM * np.ones(self.m)]),
                               np.concatenate([self.mcf.u, np.inf * np.ones(self.m)]))
        # end points of the artificial arcs are known: node i -> artificial node m where sign = +1, else m -> i
        node = np.arange(self.m, dtype=np.int64)
        self._host_arcs_of = self.mcf.A
        self._host_tail = np.concatenate([tail, np.where(sign > 0, node, self.m)])
        self._host_head = np.concatenate([head, np.where(sign > 0, self.m, node)])
        new_ids = np.arange(self.n, self.n + self.m, dtype=np.int64)
        self.artificial_vars = new_ids.astype(int)
        self.var_info["non_fix"] = np.append(self.var_info["non_fix"], new_ids)

    def rescale_cost(self, factor: float) -> None:
        """c <- c / factor.  Like the reference (:282) this rebinds `mcf.c` on the caller's object."""
        self.mcf.c = self.mcf.c / factor
        self.c_rescaling_factor = factor

    def recover_obj_val(self, obj_val: float) -> float:
        return obj_val * self.c_rescaling_factor

    def fix_variables(self, ind_fix_to_low: np.ndarray, ind_fix_to_up: np.ndarray) -> None:
        """Reference :224-234; `non_fix` / `fix` are the sorted complements (what `np.setdiff1d` returns there),
        taken with a mask instead of two sorts of n ids."""
        n = len(self.mcf.c)
        fixed = np.zeros(n, dtype=bool)
        fixed[np.asarray(ind_fix_to_low, dtype=np.int64)] = True
        fixed[np.asarray(ind_fix_to_up, dtype=np.int64)] = True
        self.var_info["fix_low"] = ind_fix_to_low
        self.var_info["fix_up"] = ind_fix_to_up
        self.var_info["non_fix"] = np.flatnonzero(~fixed)
        self.var_info["fix"] = np.flatnonzero(fixed)
        self._freed = None

    def add_free_variables(self, ind_free_new: np.ndarray) -> None:
        """Append the new columns in queue order and drop them from the fixed sets (reference :236-245).  The
        reference does three `np.setdiff1d` (sorts of the remaining fixed ids) per round; the fixed sets are
        sorted and duplicate free, so a mask of the freed arcs gives the same arrays in O(|set|)."""
        new = np.asarray(ind_free_new, dtype=np.int64)
        self.var_info["non_fix"] = np.append(self.var_info["non_fix"], ind_free_new)
        if self._freed is None or self._freed.size != self.mcf.c.size:
            self._freed = np.zeros(self.mcf.c.size, dtype=bool)
        self._freed[new] = True
        for key in ("fix", "fix_low", "fix_up"):
            arr = np.asarray(self.var_info[key])
            self.var_info[key] = arr[~self._freed[arr]] if arr.size else arr

    def set_initial_basis(self) -> None:
        vbasis = np.concatenate((-np.ones(self.n), np.zeros(self.m)))
        vbasis[self.var_info["fix_up"]] = -2
        self.set_basis(Basis(vbasis, np.concatenate([-np.ones(self.m), np.zeros(1)])))

    def set_basis(self, basis: Basis) -> None:
        self.basis = basis

    def update_subproblem(self) -> None:
        """Restricted master over the open columns, in `non_fix` order (reference :202-209), assembled from
        the arcs' end points instead of slicing the full incidence matrix: column k has +1 at tail_k and -1
        at head_k (rows ascending inside a column, the canonical form `A[:, non_fix]` has too), and the flow
        of the arcs fixed at their upper bound is moved to the right-hand side by one signed accumulation in
        ascending arc order -- the order SciPy's `A[:, up] @ u[up]` adds in, so b is bit-identical."""
        tail, head = self._host_arcs()
        nf = np.asarray(self.var_info["non_fix"], dtype=np.int64)
        up = np.asarray(self.var_info["fix_up"], dtype=np.int64)
        N, k = self.mcf.b.size, nf.size
        t, h = tail[nf], head[nf]
        rows = np.empty(2 * k, dtype=np.int64)
        vals = np.empty(2 * k)
        first = t < h
        rows[0::2] = np.where(first, t, h)
        rows[1::2] = np.where(first, h, t)
        vals[0::2] = np.where(first, 1.0, -1.0)
        vals[1::2] = -vals[0::2]
        A_sub = sp.csc_matrix((vals, rows, np.arange(0, 2 * k + 1, 2, dtype=np.int64)), shape=(N, k))
        idx = np.empty(2 * up.size, dtype=np.int64)
        w = np.empty(2 * up.size)
        idx[0::2], idx[1::2] = tail[up], head[up]
        w[0::2], w[1::2] = self.mcf.u[up], -self.mcf.u[up]
        moved = np.bincount(idx, weights=w, minlength=N) if up.size else np.zeros(N)
        self.mcf_sub = MinCostFlow(A=A_sub, b=self.mcf.b - moved, c=self.mcf.c[nf], u=self.mcf.u[nf])

    def solve_subproblem(self, solver: str, solver_settings: SolverSettings) -> Output:
        method = "network_simplex" if solver == "CPL" else "default"
        warm = Basis(self.basis.vbasis[self.var_info["non_fix"]], self.basis.cbasis)
        return solve_mcf(self.mcf_sub, solver=solver, method=method, warm_start_basis=warm, settings=solver_settings)

    def recover_x_from_sub_x(self, x_sub: np.ndarray) -> np.ndarray:
        x = np.zeros(self.mcf.c.size)
        x[self.var_info["non_fix"]] = x_sub
        x[self.var_info["fix_up"]] = self.mcf.u[self.var_info["fix_up"]]
        return x

    def recover_basis_from_sub_basis(self, basis_sub: Basis) -> Basis:
        vbasis = -np.ones(self.mcf.c.size, dtype=int)
        vbasis[self.var_info["non_fix"]] = basis_sub.vbasis
        vbasis[self.var_info["fix_up"]] = -2
        return Basis(vbasis, basis_sub.cbasis)

    # ---- K4 ------------------------------------------------------------------------------------------------------
    def price(self, y: np.ndarray, K: int = 0, want_rc: bool = False):
        """Arc-list pricing: rc_k = c_k - (y_tail - y_head), negated for arcs at their upper bound.
        The arc list, the costs, the basis statuses and the pricing buffers stay on the device between
        calls: a pass uploads the duals, and the statuses only when `set_basis` changed them."""
        import torch
        dev = _dev()
        arcs = self._device_arcs()
        vb = None
        basis = getattr(self, "basis", None)
        if basis is not None:
            if self._vb_src is not basis.vbasis:
                self._vb_dev = _cuda(np.asarray(basis.vbasis).astype(np.int8))
                self._vb_src = basis.vbasis
            vb = self._vb_dev
        pr = self._arc_pricers.get(K)
        if pr is None:
            pr = self._arc_pricers[K] = dev.Pricer(arcs["c"].device, K, fused=False)
        return dev.price_arcs(arcs["c"], arcs["tail"], arcs["head"], _cuda(np.asarray(y, dtype=np.float64)), vbasis=vb,
                              K=K, tol=TOLERANCE_FOR_REDUCED_COSTS, want_rc=want_rc, pricer=pr)

    def get_reduced_cost_for_original_mcf(self, y: np.ndarray) -> np.ndarray:
        """Reference :293-304."""
        return self.price(y, K=0, want_rc=True).rc.cpu().numpy()

    def check_optimality_condition(self, x: np.ndarray, y: np.ndarray) -> bool:
        """Reference :306-319."""
        art_ok = bool(np.all(x[self.artificial_vars] < TOLERANCE_FOR_ARTIFICIAL_VARS)) \
            if self.artificial_vars.size > 0 else True
        return bool(art_ok and self.price(y, K=0).optimal)

"""Sinkhorn warm start over row-sharded cost slabs (`sx_sinkhorn_ot_sharded_h`, `warm_start.sinkhorn` with a
`device.CostSlabs`).  One shard gives the single-GPU path's results bit for bit; G shards on one GPU (repeated
device entries) match the Sinkhorn-Knopp oracle; shards on distinct GPUs give the emulated run's results bit for
bit."""
import ctypes

import numpy as np
import pytest

import cases
from oracle import network_oracle as orc

torch = pytest.importorskip("torch")


def _n_gpus():
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


def test_sharded_entry_rejects_bad_arguments_without_gpu():
    """Null pointers and inconsistent shapes / bounds / parameters return SX_ERR_INVALID before any CUDA call."""
    from smart_crossover._native import lib
    S, D, G = 6, 5, 2
    devs = (ctypes.c_int * G)(0, 0)
    slabs = (ctypes.c_void_p * G)(16, 32)
    a, b = np.full(S, 1.0 / S), np.full(D, 1.0 / D)
    f, g = np.empty(S), np.empty(D)

    def call(ndev=G, devs_=devs, slabs_=slabs, bounds=None, ld=D, S_=S, D_=D, a_=a.ctypes.data, b_=b.ctypes.data,
             reg=0.1, max_iter=10, f_=f.ctypes.data, g_=g.ctypes.data, x_out=None):
        return lib.sx_sinkhorn_ot_sharded_h(ndev, devs_, slabs_, bounds, ld, S_, D_, a_, b_, reg, max_iter, 0.0, 10,
                                            f_, g_, x_out, None, None)

    b64 = lambda *v: (ctypes.c_int64 * len(v))(*v)
    assert call(ndev=0) == -1
    assert call(devs_=None) == -1
    assert call(slabs_=None) == -1
    assert call(slabs_=(ctypes.c_void_p * G)(16, None)) == -1
    assert call(a_=None) == -1 and call(b_=None) == -1
    assert call(f_=None) == -1 and call(g_=None) == -1
    assert call(x_out=(ctypes.c_void_p * G)(64, None)) == -1
    assert call(S_=0) == -1 and call(D_=0) == -1
    assert call(ld=D - 1) == -1
    assert call(ndev=S + 1, devs_=(ctypes.c_int * (S + 1))(), slabs_=(ctypes.c_void_p * (S + 1))(*[16] * (S + 1))) == -1
    assert call(reg=0.0) == -1 and call(reg=float("nan")) == -1
    assert call(max_iter=-1) == -1
    assert call(bounds=b64(0, 3, 5)) == -1              # does not end at S
    assert call(bounds=b64(1, 3, 6)) == -1              # does not start at 0
    assert call(bounds=b64(0, 0, 6)) == -1              # empty shard
    assert call(bounds=b64(0, 4, 3)) == -1              # decreasing


def _slabs(M, devices, bounds=None):
    from smart_crossover import device as dev
    S, D = M.shape
    sl = dev.CostSlabs(S, D, devices, bounds)
    for g in range(len(devices)):
        r0 = sl.row0[g]
        sl.view(g).copy_(torch.from_numpy(np.ascontiguousarray(M[r0:r0 + sl.rows[g]])))
    sl.sync()
    return sl


def _bits(x):
    return np.ascontiguousarray(x).tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("S,D,reg,iters,integer", [(1, 37, 0.05, 50, False), (257, 131, 0.02, 300, False),
                                                    (300, 1000, 10.0, 200, True)])
def test_one_shard_matches_single_gpu_path_bit_for_bit(S, D, reg, iters, integer):
    """G = 1: f, g and the plan are byte-for-byte those of `sinkhorn(a, b, M)` (odd D: the slab's ld is padded)."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from smart_crossover.warm_start import sinkhorn
    s, d, M = cases.ot_points(S, D, 70 + S)
    if integer:
        M = np.round(50 * M)
    X_ref, info_ref = sinkhorn(s, d, M, reg, numItermax=iters, stopThr=0.0, log=True)
    sl = _slabs(M, [torch.cuda.current_device()])
    X, info = sinkhorn(s, d, sl, reg, numItermax=iters, stopThr=0.0, log=True)
    assert info["niter"] == info_ref["niter"] == iters
    assert _bits(info["f"]) == _bits(info_ref["f"])
    assert _bits(info["g"]) == _bits(info_ref["g"])
    assert _bits(X) == _bits(X_ref)


# Row bounds of the emulated runs: equal shares and uneven ones with a 1-row shard and cuts off the 128-row chunks.
_BOUNDS = {
    2: [None, [0, 1, 257]],
    3: [None, [0, 129, 130, 257]],
    5: [None, [0, 3, 131, 200, 256, 257]],
    8: [None, [0, 1, 2, 77, 128, 129, 200, 255, 257]],
}


@pytest.mark.gpu
@pytest.mark.parametrize("G,bi", [(G, i) for G in (2, 3, 5, 8) for i in range(2)])
def test_emulated_shards_match_sinkhorn_knopp(G, bi):
    """G ranks on one GPU: plan == oracle to 1e-9, rows meet `a`, and the stopping rule stops within one
    iteration of the oracle's."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from smart_crossover.warm_start import sinkhorn
    S, D, reg, iters = 257, 130, 0.02, 500
    s, d, M = cases.ot_points(S, D, 40 + S)
    bounds = _BOUNDS[G][bi]
    sl = _slabs(M, [torch.cuda.current_device()] * G, bounds)
    X_ref, _, _ = orc.sinkhorn_knopp(s, d, M, reg, iters, stop_thr=0.0)
    X, info = sinkhorn(s, d, sl, reg, numItermax=iters, stopThr=0.0, log=True)
    assert info["niter"] == iters and X.shape == (S, D)
    np.testing.assert_allclose(X, X_ref, rtol=1e-9, atol=1e-300)
    np.testing.assert_allclose(X.sum(axis=1), s, rtol=1e-9)
    X2, info2 = sinkhorn(s, d, sl, reg, numItermax=10000, stopThr=1e-7, log=True)
    _, it2, _ = orc.sinkhorn_knopp(s, d, M, reg, 10000, stop_thr=1e-7)
    assert info2["err"] < 1e-7 and abs(info2["niter"] - it2) <= 1


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, "all"])
def test_distinct_devices_match_the_emulation_bit_for_bit(n):
    """Shards on distinct GPUs (NVLink exchange) == the same row bounds emulated on one GPU, byte for byte -- the
    stopping error too: the fold's per-CTA error sums are added in CTA order, not by atomics."""
    n_vis = _n_gpus()
    if n_vis < 2:
        pytest.skip("needs at least 2 GPUs")
    from smart_crossover.warm_start import sinkhorn
    G = n_vis if n == "all" else 2
    S, D, reg = 1000, 777, 0.02
    s, d, M = cases.ot_points(S, D, 4711)
    bounds = [0] + sorted(np.random.default_rng(G).choice(np.arange(1, S), G - 1, replace=False).tolist()) + [S]
    runs = []
    for devices in ([0] * G, list(range(G))):
        sl = _slabs(M, devices, bounds)
        runs.append(sinkhorn(s, d, sl, reg, numItermax=2000, stopThr=1e-8, log=True))
    (Xe, ie), (Xd, idv) = runs
    assert ie["niter"] == idv["niter"] and ie["err"] == idv["err"]
    assert _bits(ie["f"]) == _bits(idv["f"]) and _bits(ie["g"]) == _bits(idv["g"])
    assert _bits(Xe) == _bits(Xd)


@pytest.mark.gpu
def test_device_resident_problem_warm_starts_from_its_slabs():
    """`sinkhorn(s, d, slabs)` on the slabs of an `OTManager.from_device_cost` manager: the host M is never read."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from smart_crossover.network_methods.net_manager import OTManager
    from smart_crossover.warm_start import sinkhorn
    S, D, reg, iters = 200, 150, 0.05, 300
    s, d, M = cases.ot_points(S, D, 99)
    cur = torch.cuda.current_device()
    slabs = _slabs(M, [cur, cur], [0, 90, S])
    mgr = OTManager.from_device_cost(s, d, slabs)
    with pytest.raises(TypeError):
        np.asarray(mgr.ot.M)                              # no host copy to fall back on
    X, info = sinkhorn(mgr.ot.s, mgr.ot.d, slabs, reg, numItermax=iters, stopThr=0.0, log=True)
    X_ref, _, _ = orc.sinkhorn_knopp(s, d, M, reg, iters, stop_thr=0.0)
    assert info["niter"] == iters
    np.testing.assert_allclose(X, X_ref, rtol=1e-9, atol=1e-300)

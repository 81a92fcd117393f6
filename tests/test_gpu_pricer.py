"""The persistent pricer behind the managers (`sx_ot_pricer`, include/sxcross.h) and the one-shot host-buffer
entry point `sx_price_dense_ot_h`, called with NumPy buffers exactly as a binding inside the reference's
`OTManager.check_optimality_condition` (net_manager.py:485-497) would, against the CPU oracle.
Multi-device cases need >= 2 GPUs in ONE process (no torchrun) and are skipped otherwise."""
import ctypes
import os
import re

import numpy as np
import pytest

import cases
from golden_util import OT_FULL, Fixture
from oracle import network_oracle as orc

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from smart_crossover import device
    return device


def n_gpus():
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


def check_pass(res, M, y, K):
    S = M.shape[0]
    rc = orc.reduced_costs_ot(M, y)
    cnt, mn, ids, vals = orc.price_summary(rc, K)
    assert res.n_violating == cnt and res.min_rc == mn
    assert np.array_equal(res.topk_id, ids) and res.topk_rc.tobytes() == vals.tobytes()
    assert res.optimal == bool(np.all(rc >= -1e-6))


def pass_list(M, seed):
    S, D = M.shape
    return [cases.planted_duals(M, seed, 0.05), cases.planted_duals(M, seed + 1, 0.3),
            cases.planted_duals(M, seed + 2, 0.0) - np.concatenate([np.zeros(S), np.full(D, 1e-3)]),
            np.concatenate([np.zeros(S), np.full(D, 5.0)]), cases.planted_duals(M, seed + 3, 0.01)]


@pytest.mark.parametrize("S,D", [(1, 1), (40, 40), (257, 513), (1000, 1002)])
@pytest.mark.parametrize("K", [0, 1, 100, 1024, 3000])
def test_ot_pricer_one_device(dev, S, D, K):
    """Odd D is padded to an even leading dimension by CostSlabs, so these all take the fused kernel
    (K = 3000 > SX_TOPK_MAX_K: separate kernels + sorted selection)."""
    s, d, M = cases.ot_points(S, D, 300 + S)
    pr = dev.OTPricer(dev.CostSlabs.from_host(M, [torch.cuda.current_device()]), K)
    assert pr.stats()["fused"] == (K <= 1024)
    for rep in range(2):
        for y in pass_list(M, 5):
            check_pass(pr.price(y[:S], y[S:]), M, y, K)
    assert pr.stats()["passes"] == 10
    pr.close()


def test_ot_pricer_repeats_only_after_overflow(dev):
    """1.56 M arcs with the SAME reduced cost: nothing can be pruned, the candidate buffer (2^20) overflows
    -> grown and priced again; the 1.56 M candidates that tie at the K-th value are refined on the arc id
    inside the fused pass.  All inside one sx_ot_pricer_price_h call; the second call does not repeat."""
    S, D, K = 1200, 1300, 100
    M = np.full((S, D), 2.0)
    y = np.concatenate([np.zeros(S), np.full(D, 3.0)])
    pr = dev.OTPricer(dev.CostSlabs.from_host(M, [torch.cuda.current_device()]), K)
    for _ in range(2):
        res = pr.price(y[:S], y[S:])
        assert res.n_violating == S * D and res.min_rc == -1.0
        assert np.array_equal(res.topk_id, np.arange(K)) and np.all(res.topk_rc == -1.0)
    st = pr.stats()
    assert st["repeated_passes"] == 1
    y2 = cases.planted_duals(M + np.random.default_rng(0).random((S, D)), 3, 0.1)      # an ordinary pass afterwards
    M2 = M.copy()
    check_pass(pr.price(y2[:S], y2[S:]), M2, y2, K)
    pr.close()


def test_ot_pricer_nan_is_not_optimal(dev):
    S, D = 64, 128
    s, d, M = cases.ot_points(S, D, 9)
    y = cases.planted_duals(M, 9, 0.0)
    y[S:] -= 1e-3
    pr = dev.OTPricer(dev.CostSlabs.from_host(M, [torch.cuda.current_device()]), 0)
    assert pr.price(y[:S], y[S:]).optimal
    y[3] = np.nan
    res = pr.price(y[:S], y[S:])
    assert res.n_violating == 0 and res.has_nan and not res.optimal


@pytest.mark.parametrize("name", OT_FULL)
def test_one_shot_host_entry_point_with_numpy_buffers(dev, name):
    """sx_price_dense_ot_h, the entry a reference-side binding calls with NumPy arrays (round-1 stub)."""
    from smart_crossover._native import check, lib
    fx = Fixture(name)
    M = np.ascontiguousarray(fx.inp["M"], dtype=np.float64)
    S, D = M.shape
    K = 32
    for tag in ("tree", "pert"):
        y = np.ascontiguousarray(fx.out["y_" + tag], dtype=np.float64)
        cnt, mn = ctypes.c_ulonglong(0), ctypes.c_double(0)
        rc_k, id_k, n_k = np.empty(K), np.empty(K, dtype=np.int64), ctypes.c_int64(0)
        check(lib.sx_price_dense_ot_h(M.ctypes.data, None, S, D, y.ctypes.data, 1e-6, K, ctypes.byref(cnt),
                                      ctypes.byref(mn), rc_k.ctypes.data, id_k.ctypes.data, ctypes.byref(n_k)), "h")
        rc_ref = fx.out["rc_" + tag]
        c_ref, m_ref, ids, vals = orc.price_summary(rc_ref, K)
        assert cnt.value == c_ref and mn.value == m_ref and n_k.value == ids.size
        assert np.array_equal(id_k[:ids.size], ids) and rc_k[:ids.size].tobytes() == vals.tobytes()
        assert (cnt.value == 0) == bool(fx.out["optimal_" + tag])
        # device-resident matrix from an earlier upload (leading dimension D) gives the same
        Md = torch.from_numpy(M).cuda()
        cnt2 = ctypes.c_ulonglong(0)
        check(lib.sx_price_dense_ot_h(None, ctypes.c_void_p(Md.data_ptr()), S, D, y.ctypes.data, 1e-6, 0,
                                      ctypes.byref(cnt2), ctypes.byref(mn), None, None, None), "h dev")
        assert cnt2.value == c_ref


def test_integration_md_binding_stub_runs_verbatim(dev):
    """INTEGRATION.md section B shows the binding a reference maintainer would add; the code block is
    executed here as written and its class is driven like `column_generation` drives the manager."""
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    m = re.search(r"<!-- binding-stub-begin -->\s*```python\n(.*?)```\s*<!-- binding-stub-end -->", text, re.S)
    assert m, "INTEGRATION.md lost its binding stub markers"
    ns = {"SXCROSS_LIB": os.path.join(ROOT, "smart-crossover_b200", "libsxcross.so")}
    exec(compile(m.group(1), "INTEGRATION.md#B", "exec"), ns)
    fx = Fixture("ot_c1_40x40")
    M = fx.inp["M"]
    pricer = ns["DevicePricing"](M)
    for tag in ("tree", "pert"):
        assert pricer.all_reduced_costs_nonnegative(fx.out["y_" + tag]) == bool(fx.out["optimal_" + tag])
    pricer.close()


# ---- several GPUs, ONE process ---------------------------------------------------------------------------
@pytest.mark.skipif(n_gpus() < 2, reason="needs at least 2 GPUs")
@pytest.mark.parametrize("K", [0, 64, 1024])
@pytest.mark.parametrize("S,D", [(301, 518), (64, 4097), (2000, 3000)])
def test_ot_pricer_all_devices_one_process(dev, S, D, K):
    G = min(n_gpus(), 8, S)
    s, d, M = cases.ot_points(S, D, 700 + S)
    pr = dev.OTPricer(dev.CostSlabs.from_host(M, list(range(G))), K)
    st = pr.stats()
    assert st["fused"] and st["merge_in_kernel"] and st["devices"] == list(range(G))
    for rep in range(2):
        for y in pass_list(M, 8):
            check_pass(pr.price(y[:S], y[S:]), M, y, K)
    pr.close()


@pytest.mark.skipif(n_gpus() < 2, reason="needs at least 2 GPUs")
def test_ot_pricer_uneven_shards(dev):
    """Shards sized by the caller (`row_bounds`, as `balanced_row_bounds` produces them): same answers."""
    G = min(n_gpus(), 8)
    S, D, K = 16 * G + 37, 1030, 128
    s, d, M = cases.ot_points(S, D, 55)
    bounds = [0] + sorted(np.random.default_rng(3).choice(np.arange(1, S), G - 1, replace=False).tolist()) + [S]
    pr = dev.OTPricer(dev.CostSlabs.from_host(M, list(range(G)), row_bounds=bounds), K)
    for y in pass_list(M, 2):
        check_pass(pr.price(y[:S], y[S:]), M, y, K)
    pr.close()
    with pytest.raises(ValueError):
        dev.CostSlabs(S, D, list(range(G)), row_bounds=[0] * G + [S])


@pytest.mark.skipif(n_gpus() < 2, reason="needs at least 2 GPUs")
def test_ot_pricer_multi_device_overflow_repeat_protocol(dev):
    """Every device's candidate buffer (2^20) overflows at once (1.43 M tied arcs each): all ranks grow it and
    repeat together, once; the ties are then refined inside the fused pass."""
    G = min(n_gpus(), 8)
    S, D, K = 1100 * G, 1300, 100
    M = np.full((S, D), 2.0)
    y = np.concatenate([np.zeros(S), np.full(D, 3.0)])
    pr = dev.OTPricer(dev.CostSlabs.from_host(M, list(range(G))), K)
    for _ in range(2):
        res = pr.price(y[:S], y[S:])
        assert res.n_violating == S * D and np.array_equal(res.topk_id, np.arange(K))
    assert pr.stats()["repeated_passes"] == 1
    rng = np.random.default_rng(1)
    M2 = rng.random((S, D))
    pr2 = dev.OTPricer(dev.CostSlabs.from_host(M2, list(range(G))), K)
    y2 = cases.planted_duals(M2, 4, 0.1)
    check_pass(pr2.price(y2[:S], y2[S:]), M2, y2, K)


@pytest.mark.skipif(n_gpus() < 2, reason="needs at least 2 GPUs")
@pytest.mark.parametrize("method", ["tnet", "cnet_ot"])
def test_network_crossover_prices_on_every_gpu(dev, method, monkeypatch):
    """`network_crossover` (algorithms.py:14-78) as a plain function call with SX_DEVICES=all: the manager's
    pricer shards the cost matrix over every GPU of the box; objective / basis equal the reference's."""
    from smart_crossover.formats import OptTransport
    from smart_crossover.network_methods import net_manager
    from smart_crossover.network_methods.algorithms import network_crossover
    from smart_crossover.solver_caller.caller import SolverSettings
    monkeypatch.setenv("SX_DEVICES", "all")
    seen = []
    orig = net_manager.OTManager._device_slabs

    def spy(self):
        slabs = orig(self)
        seen.append(tuple(slabs.devices))
        return slabs
    monkeypatch.setattr(net_manager.OTManager, "_device_slabs", spy)
    fx = Fixture("ot_c1_40x40")
    ot = OptTransport(fx.inp["s"], fx.inp["d"], fx.inp["M"])
    out = network_crossover(fx.inp["x"], ot=ot, method=method, solver="HGS", solver_settings=SolverSettings(log_console=0))
    assert seen and len(seen[0]) == min(n_gpus(), 40 if method == "tnet" else 41)
    ref = float(fx.out[method + "_obj"])
    assert abs(out.obj_val - ref) <= 1e-9 * abs(ref)
    assert np.array_equal(np.flatnonzero(out.basis.vbasis == 0), fx.out[method + "_basic"])
    assert out.iter_count == int(fx.out[method + "_iters"])

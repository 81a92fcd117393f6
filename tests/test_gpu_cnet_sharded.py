"""CNET_OT on a device-resident, row-sharded OT problem: the big-M extension priced over the base slabs
(`sx_price_dense_ot_fused_bigm`, `sx_ot_pricer_create_bigm`) must give what the physically extended matrix gives,
bit for bit -- count, minimum, NaN status, top-K ids and values -- and `network_crossover(method="cnet_ot")` on a
`DeviceResidentCost` must follow the host route's path."""
import ctypes

import numpy as np
import pytest

import cases
from golden_util import Fixture
from oracle import network_oracle as orc

torch = pytest.importorskip("torch")

SX_ERR_INVALID, SX_ERR_TOO_LARGE, SX_ERR_UNALIGNED = -1, -4, -6


def _n_gpus():
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


def _need_cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


# ---- without a GPU -------------------------------------------------------------------------------------------------
def test_fused_bigm_entry_rejects_bad_arguments_without_gpu():
    """Null pointers, bad bounds, a shard past S, odd ld and K > SX_TOPK_MAX_K fail before any CUDA call."""
    from smart_crossover._native import lib
    S, D = 40, 30

    def call(M=16, ld=32, row0=0, S_loc=S, S_=S, D_=D, y_src=32, y_dst=48, y_art=64, state=80, K=4, block=96,
             block_len=64, ws=112):
        return lib.sx_price_dense_ot_fused_bigm(M, ld, None, 0, row0, S_loc, S_, D_, y_src, y_dst, y_art, 1e3, 0.0,
                                                1e-6, state, None, None, 0, K, block, block_len, None, 0, 1, None,
                                                None, ws, 1 << 40, None)

    for kw in ({"M": None}, {"y_src": None}, {"y_dst": None}, {"state": None}, {"block": None}):
        assert call(**kw) == SX_ERR_INVALID, kw
    assert call(ws=None) == -3                                     # SX_ERR_WORKSPACE
    assert call(y_art=None) == SX_ERR_INVALID                      # the shard ends at S: u_S is needed
    assert call(S_loc=0) == SX_ERR_INVALID and call(row0=-1) == SX_ERR_INVALID
    assert call(S_=0) == SX_ERR_INVALID and call(D_=0) == SX_ERR_INVALID
    assert call(row0=10, S_loc=31) == SX_ERR_INVALID               # row0 + S_loc > S
    assert call(row0=0, S_loc=S + 1) == SX_ERR_INVALID
    assert call(ld=D - 2) == SX_ERR_INVALID                        # ld < D
    assert call(ld=31) == SX_ERR_UNALIGNED                         # odd ld: no TMA path
    assert call(M=24) == SX_ERR_UNALIGNED
    assert call(K=1025) == SX_ERR_INVALID and call(K=0) == SX_ERR_INVALID
    assert call(block_len=2 * 4 + 5) == SX_ERR_INVALID
    assert call(D_=(1 << 31) - 1, ld=1 << 31) == SX_ERR_TOO_LARGE   # D + 1 = 2^31: ids of a row do not fit


def test_bigm_pricer_create_rejects_bad_arguments_without_gpu():
    from smart_crossover._native import lib
    S, D, G = 6, 5, 2
    h = ctypes.c_void_p()
    b64 = lambda *v: (ctypes.c_int64 * len(v))(*v)

    def call(ndev=G, devs=(ctypes.c_int * G)(0, 0), slabs=(ctypes.c_void_p * G)(16, 32), bounds=None, ld=6, S_=S,
             D_=D, K=4, out=ctypes.byref(h)):
        return lib.sx_ot_pricer_create_bigm(ndev, devs, slabs, bounds, ld, S_, D_, 1e3, 0.0, K, 1e-6, out)

    assert call(out=None) == SX_ERR_INVALID
    assert call(ndev=0) == SX_ERR_INVALID and call(devs=None) == SX_ERR_INVALID and call(slabs=None) == SX_ERR_INVALID
    assert call(slabs=(ctypes.c_void_p * G)(16, None)) == SX_ERR_INVALID
    assert call(S_=0) == SX_ERR_INVALID and call(D_=0) == SX_ERR_INVALID and call(ld=4) == SX_ERR_INVALID
    assert call(K=-1) == SX_ERR_INVALID
    assert call(bounds=b64(0, 3, 5)) == SX_ERR_INVALID             # does not end at S
    assert call(bounds=b64(1, 3, 6)) == SX_ERR_INVALID             # does not start at 0
    assert call(bounds=b64(0, 0, 6)) == SX_ERR_INVALID             # empty shard
    assert call(ndev=1, devs=(ctypes.c_int * 1)(0), slabs=(ctypes.c_void_p * 1)(16), ld=7) == SX_ERR_UNALIGNED
    assert call(slabs=(ctypes.c_void_p * G)(16, 40)) == SX_ERR_UNALIGNED
    assert call(ndev=1, devs=(ctypes.c_int * 1)(0), slabs=(ctypes.c_void_p * 1)(16), K=1025) == SX_ERR_TOO_LARGE
    assert call(K=1025) == SX_ERR_TOO_LARGE
    assert h.value is None


class _StubSlabs:
    """What `DeviceResidentCost` reads of `device.CostSlabs`, over a host matrix."""

    def __init__(self, M):
        self.M = M
        self.S, self.D = M.shape
        self.max_calls = 0

    def take_flat(self, ids):
        return self.M.ravel()[np.asarray(ids, dtype=np.int64)]

    def max(self):
        self.max_calls += 1
        return float(np.max(self.M))


def test_device_resident_max_and_bigm_view_over_a_stub():
    from smart_crossover.network_methods.net_manager import BigMExtendedCost, DeviceResidentCost
    S, D = 7, 5
    M = np.random.default_rng(1).random((S, D))
    stub = _StubSlabs(M)
    cost = DeviceResidentCost(stub)
    assert np.max(cost) == M.max() and stub.max_calls == 1         # np.max dispatches to .max(axis=None, out=None)
    with pytest.raises(ValueError):
        np.max(cost, axis=0)
    with pytest.raises(TypeError, match="device resident"):
        np.asarray(cost)
    bigM = 123.0
    ext = BigMExtendedCost(cost, bigM)
    host = BigMExtendedCost(M, bigM)
    assert ext.shape == host.shape == (S + 1, D + 1) and ext.size == (S + 1) * (D + 1)
    border = np.concatenate([np.arange(S) * (D + 1) + D, S * (D + 1) + np.arange(D + 1)])
    inner = np.array([0, 3, (D + 1) + 2, (S - 1) * (D + 1) + D - 1])
    for ids in (border, inner, np.concatenate([inner, border[::-1]])):
        assert ext.take_flat(ids).tobytes() == host.take_flat(ids).tobytes()
    assert ext.take_flat(border[:-1]).tolist() == [bigM] * (S + D) and ext.take_flat(border[-1:]).tolist() == [0.0]
    with pytest.raises(TypeError, match="device resident"):
        np.asarray(ext)
    assert np.max(ext) == bigM and np.max(host) == bigM


# ---- on one GPU ------------------------------------------------------------------------------------------------------
def _extend(M, bigM, corner=0.0):
    S, D = M.shape
    X = np.full((S + 1, D + 1), bigM)
    X[:S, :D] = M
    X[S, D] = corner
    return X


def _dual_sets(M, bigM, integer=False):
    """Duals of the (S+1) x (D+1) extension, in the order a column generation might meet them: sparse, dense, sparse
    (both walks of the fused pass run)."""
    S, D = M.shape
    X = _extend(M, bigM)
    ys = {}
    ys["planted"] = cases.planted_duals(X, 3, 0.05)
    ys["converged"] = cases.planted_duals(X, 4, 0.0)
    y = cases.planted_duals(M, 5, 0.0)                              # the base's converged duals ...
    ys["border_only"] = np.concatenate([y[:S], [-bigM - 3.0], y[S:], [bigM + y[:S].max() + 2.0]])   # ... u_S, v_D violate
    ys["all"] = np.concatenate([np.zeros(S + 1), np.full(D + 1, bigM + M.max() + 1.0)])
    ys["sparse_again"] = cases.planted_duals(X, 6, 0.01)
    for what, at in (("nan_u_S", S), ("nan_v_D", S + 1 + D), ("nan_inner", 2)):
        y = cases.planted_duals(X, 7, 0.02)
        y[at] = np.nan
        ys[what] = y
    if integer:                                                     # exact ties between border and inner arcs
        rng = np.random.default_rng(8)
        for n in range(2):
            ys[f"ties{n}"] = np.concatenate([rng.integers(0, 3, S + 1), rng.integers(3, 9, D + 1)]).astype(np.float64)
    return ys


def _same(a, b):
    assert a.n_violating == b.n_violating
    assert np.float64(a.min_rc).tobytes() == np.float64(b.min_rc).tobytes()
    assert a.status == b.status
    assert np.array_equal(a.topk_id, b.topk_id) and a.topk_rc.tobytes() == b.topk_rc.tobytes()


def _check_oracle(res, X, y, K):
    cnt, mn, ids, vals = orc.price_summary(orc.reduced_costs_ot(X, y), K)
    assert res.n_violating == cnt
    if not np.isnan(y).any():
        assert res.min_rc == mn
    if K:
        assert np.array_equal(res.topk_id, ids) and res.topk_rc.tobytes() == vals.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("K", [0, 1, 64, 1024])
@pytest.mark.parametrize("S,D", [(S, D) for S in (15, 16, 17) for D in (255, 256, 257)])
def test_bigm_pricer_equals_the_extended_matrix(S, D, K):
    _need_cuda()
    from smart_crossover import _native
    from smart_crossover import device as dev
    cur = torch.cuda.current_device()
    integer = (S + D) % 2 == 0
    if integer:
        M = np.random.default_rng(S * D).integers(0, 10, (S, D)).astype(np.float64)
        bigM = 7.0
    else:
        M = cases.ot_points(S, D, S * D)[2]
        bigM = float((S + D) * M.max())
    base = dev.CostSlabs.from_host(M, [cur])
    ext = dev.CostSlabs.from_host(M, [cur], border=(bigM, 0.0))
    pb = dev.OTPricer(base, K, bigm=(bigM, 0.0))
    pe = dev.OTPricer(ext, K)
    assert pb.stats()["fused"] and pe.stats()["fused"]
    X = _extend(M, bigM)
    for name, y in _dual_sets(M, bigM, integer).items():
        a = pb.price(y[:S + 1], y[S + 1:])
        b = pe.price(y[:S + 1], y[S + 1:])
        _same(a, b)
        _check_oracle(a, X, y, K)
        if name.startswith("nan"):
            assert a.status & _native.SX_STATUS_NAN_RC and not a.optimal
        if name == "border_only":
            assert a.n_violating > 0 and np.all((a.topk_id % (D + 1) == D) | (a.topk_id // (D + 1) == S))
    with pytest.raises(ValueError):
        pb.price(np.zeros(S), np.zeros(D + 1))
    pb.close()
    pe.close()


@pytest.mark.gpu
def test_bigm_pricer_candidate_overflow_repeats():
    """Every arc of a constant matrix ties, border included: more candidates than the first buffer holds, so both
    pricers grow it and repeat; the top-K is the smallest ids."""
    _need_cuda()
    from smart_crossover import device as dev
    cur = torch.cuda.current_device()
    S, D, K = 1100, 1000, 1024
    M = np.full((S, D), 2.0)
    base = dev.CostSlabs.from_host(M, [cur])
    ext = dev.CostSlabs.from_host(M, [cur], border=(2.0, 2.0))
    pb, pe = dev.OTPricer(base, K, bigm=(2.0, 2.0)), dev.OTPricer(ext, K)
    y = np.concatenate([np.zeros(S + 1), np.full(D + 1, 3.0)])
    for _ in range(2):
        a, b = pb.price(y[:S + 1], y[S + 1:]), pe.price(y[:S + 1], y[S + 1:])
        _same(a, b)
        assert a.n_violating == (S + 1) * (D + 1) and np.array_equal(a.topk_id, np.arange(K))
    assert pb.stats()["repeated_passes"] >= 1 and pe.stats()["repeated_passes"] >= 1
    pb.close()
    pe.close()


def _uneven_last_one(S, G):
    """G + 1 row bounds, uneven, the last shard a single row."""
    if G == 1:
        return [0, S]
    cut = np.random.default_rng(G).choice(np.arange(1, S - 1), G - 2, replace=False)
    return [0] + sorted(int(v) for v in cut) + [S - 1, S]


@pytest.mark.gpu
@pytest.mark.parametrize("G,K", [(2, 128), (8, 1024), (5, 33), (3, 1)])
def test_fused_bigm_pass_pushes_to_emulated_ranks(G, K):
    """sx_price_dense_ot_fused_bigm per emulated rank on one GPU, then sx_topk_merge_ll in every rank's buffer: the
    merged block is the oracle's top-K of the explicit extension."""
    _need_cuda()
    from smart_crossover import device as dev
    from smart_crossover._native import check, lib
    S, D = 64 * G + 3, 700
    M = cases.ot_points(S, D, 70 + G)[2]
    bigM = float(M.max() * 1.5)
    X = _extend(M, bigM)
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    Mt = cu(M)
    blk = 2 * K + dev.Pricer.BLOCK_TAIL
    bufs = [torch.zeros(lib.sx_exchange_ll_buffer_bytes(blk, G) // 8, dtype=torch.int64, device="cuda")
            for _ in range(G)]
    ptrs = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device="cuda")
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    bounds = _uneven_last_one(S, G)
    assert bounds[-1] - bounds[-2] == 1
    pricers = [dev.Pricer(torch.device("cuda"), K, fused=True) for _ in range(G)]
    for name, y in _dual_sets(M, bigM).items():
        yt = cu(y)
        cnt, mn, ids, vals = orc.price_summary(orc.reduced_costs_ot(X, y), K)
        for g in range(G):
            r0, r1 = bounds[g], bounds[g + 1]
            pricers[g].price_dense_fused(Mt[r0:r1], D, r0, r1 - r0, D, yt[r0:r1], yt[S + 1:], peer_bufs=dev._ptr(ptrs),
                                         rank=g, G=G, bigm=(S, yt[S:S + 1], bigM, 0.0))
        for g in range(G):
            out = torch.zeros(2 * K + 6, dtype=torch.int64, device="cuda")
            check(lib.sx_topk_merge_ll(dev._ptr(bufs[g]), blk, G, K, dev._ptr(out[:K]), dev._ptr(out[K:2 * K]),
                                       dev._ptr(out[2 * K:]), dev._ptr(out[2 * K + 1:]), dev._ptr(status),
                                       dev._stream()), "merge_ll")
            h = out.cpu().numpy()
            k = int(h[2 * K])
            assert int(status.item()) == 0 and k == ids.size, name
            assert np.array_equal(h[K:K + k], ids) and h[:k].view(np.float64).tobytes() == vals.tobytes(), name
            assert int(h[2 * K + 1]) == cnt, name
            if not name.startswith("nan"):
                assert lib.sx_key_to_f64(int(h[2 * K + 2])) == mn, name
            assert bool(int(h[2 * K + 4]) & 8) == name.startswith("nan"), name
            assert np.all(h[K + k:2 * K] == -1)


def _managers(devices, bounds=None):
    """The 784^2 golden as a host-matrix manager and as a device-resident one, both extended by big-M."""
    from golden_util import c2_inputs
    from smart_crossover import device as dev
    from smart_crossover.formats import OptTransport
    from smart_crossover.network_methods.net_manager import DeviceResidentCost, OTManager
    s, d, M, x = c2_inputs()
    host = OTManager(OptTransport(s.copy(), d.copy(), M.copy()))
    slabs = dev.CostSlabs.from_host(M, devices, row_bounds=bounds)
    devm = OTManager(OptTransport(s.copy(), d.copy(), DeviceResidentCost(slabs)))
    bigM = host.m * np.max(M)
    assert np.max(devm.ot.M) == np.max(M)
    host.extend_by_bigM(bigM)
    devm.extend_by_bigM(host.m * np.max(devm.ot.M))
    assert devm._slabs is slabs and devm.ot.M.bigM == host.ot.M.bigM
    return host, devm, (s, d, M, x)


@pytest.mark.gpu
def test_manager_784_matches_the_host_route():
    _need_cuda()
    cur = torch.cuda.current_device()
    host, devm, (s, d, M, x) = _managers([cur])
    S, D = 784, 784
    opened = np.random.default_rng(11).choice(S * D, 3000, replace=False)      # ids of the original problem
    for mgr in (host, devm):
        mgr.add_free_variables(opened)
    a, b = host.get_sub_problem(), devm.get_sub_problem()
    assert (a.A != b.A).nnz == 0 and a.b.tobytes() == b.b.tobytes() and a.c.tobytes() == b.c.tobytes()
    X = _extend(M, host.ot.M.bigM)
    rng = np.random.default_rng(12)
    xs = [np.zeros((S + 1) * (D + 1)), np.where(rng.random((S + 1) * (D + 1)) < 0.01, 1.0, 0.0)]
    ys = [cases.planted_duals(X, 13, 0.0), cases.planted_duals(X, 14, 0.02),
          np.concatenate([cases.planted_duals(M, 15, 0.0)[:S], [0.0], cases.planted_duals(M, 15, 0.0)[S:], [0.0]])]
    for y in ys:
        rh, rd = host.get_reduced_cost_for_original_OT(y), devm.get_reduced_cost_for_original_OT(y)
        assert rh.shape == rd.shape == ((S + 1) * (D + 1),) and rh.tobytes() == rd.tobytes()
        assert rd.tobytes() == orc.reduced_costs_ot(X, y).tobytes()
        for xx in xs:
            assert host.check_optimality_condition(xx, y) == devm.check_optimality_condition(xx, y)
        for K in (0, 16):
            _same(host.price(y, K), devm.price(y, K))
    assert any(host.check_optimality_condition(xs[0], y) for y in ys)
    assert not all(host.check_optimality_condition(xs[0], y) for y in ys)


def _cnet_e2e(devices, bounds=None):
    from golden_util import c2_inputs
    from smart_crossover import device as dev
    from smart_crossover.formats import OptTransport
    from smart_crossover.network_methods.algorithms import network_crossover
    from smart_crossover.network_methods.net_manager import DeviceResidentCost
    from smart_crossover.solver_caller.caller import SolverSettings
    s, d, M, x = c2_inputs()
    fx = Fixture("e2e_c2_784")
    slabs = dev.CostSlabs.from_host(M, devices, row_bounds=bounds)
    flow = dev.CostSlabs.from_host(x, like=slabs)
    out = network_crossover(x=flow, ot=OptTransport(s.copy(), d.copy(), DeviceResidentCost(slabs)), method="cnet_ot",
                            solver="HGS", solver_settings=SolverSettings(log_console=0))
    ref = float(fx.out["cnet_ot_obj"])
    assert abs(out.obj_val - ref) <= 1e-9 * abs(ref)
    assert out.iter_count == int(fx.out["cnet_ot_iters"])
    assert np.array_equal(np.flatnonzero(out.basis.vbasis == 0), fx.out["cnet_ot_basic"])
    return out


@pytest.mark.gpu
def test_network_crossover_cnet_ot_on_device_resident_784():
    _need_cuda()
    _cnet_e2e([torch.cuda.current_device()])


# ---- on several GPUs -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, "all"])
def test_distinct_devices_match_one_device(n):
    """The bigM pricer with shards on distinct GPUs == the same problem on one GPU, and cnet_ot end to end on them."""
    n_vis = _n_gpus()
    if n_vis < 2:
        pytest.skip("needs at least 2 GPUs")
    from smart_crossover import device as dev
    G = n_vis if n == "all" else 2
    S, D, K = 1500, 1502, 256
    M = cases.ot_points(S, D, 31)[2]
    bigM = float(M.max() * 2.0)
    one = dev.OTPricer(dev.CostSlabs.from_host(M, [0]), K, bigm=(bigM, 0.0))
    many = dev.OTPricer(dev.CostSlabs.from_host(M, list(range(G))), K, bigm=(bigM, 0.0))
    assert many.stats()["devices"] == list(range(G))
    for y in _dual_sets(M, bigM).values():
        _same(one.price(y[:S + 1], y[S + 1:]), many.price(y[:S + 1], y[S + 1:]))
    one.close()
    many.close()
    _cnet_e2e(list(range(G)))

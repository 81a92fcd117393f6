"""TNET on a row-sharded, device-resident OT problem: the head of the Kruskal order / the queue selected across
shards (`sx_order_head_sharded_h`), the spanning tree and the lazy queue built from flow slabs, the Sinkhorn flow
returned as slabs, and `network_crossover` end to end.  Shards on one GPU (repeated device entries) must give the
host path's results bit for bit; shards on distinct GPUs must give the emulation's."""
import ctypes

import numpy as np
import pytest

import cases
from golden_util import Fixture
from oracle import network_oracle as orc

torch = pytest.importorskip("torch")


def _n_gpus():
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


def _need_cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def test_sharded_head_entry_rejects_bad_arguments_without_gpu():
    """Null pointers, bad bounds, S * D >= 2^32, T_cap < T and an unknown mode fail before any CUDA call."""
    from smart_crossover._native import lib
    S, D, G = 6, 5, 2
    devs = (ctypes.c_int * G)(0, 0)
    w = (ctypes.c_void_p * G)(16, 32)
    n_out = ctypes.c_int64(0)

    def call(ndev=G, devs_=devs, w_=w, bounds=None, S_=S, D_=D, T=4, T_cap=8, hist=None, mode=0, out=64,
             n_out_=ctypes.byref(n_out)):
        return lib.sx_order_head_sharded_h(ndev, devs_, w_, bounds, S_, D_, T, T_cap, hist, mode, out, n_out_)

    b64 = lambda *v: (ctypes.c_int64 * len(v))(*v)
    assert call(ndev=0) == -1
    assert call(devs_=None) == -1 and call(w_=None) == -1
    assert call(w_=(ctypes.c_void_p * G)(16, None)) == -1
    assert call(out=None) == -1 and call(n_out_=None) == -1
    assert call(S_=0) == -1 and call(D_=0) == -1
    assert call(ndev=S + 1, devs_=(ctypes.c_int * (S + 1))(), w_=(ctypes.c_void_p * (S + 1))(*[16] * (S + 1))) == -1
    assert call(T=0) == -1
    assert call(T=9, T_cap=8) == -1                     # T_cap < T
    assert call(mode=2) == -1
    assert call(bounds=b64(0, 3, 5)) == -1              # does not end at S
    assert call(bounds=b64(1, 3, 6)) == -1              # does not start at 0
    assert call(bounds=b64(0, 0, 6)) == -1              # empty shard
    assert call(bounds=b64(0, 4, 3)) == -1              # decreasing
    assert call(S_=1 << 16, D_=1 << 16) == -4           # S * D = 2^32 arcs: ids do not fit uint32
    assert call(S_=3, D_=(1 << 32) + 1) == -4


def _uneven(S, G, seed=0):
    """Row bounds with 1-row shards first, the rest cut at random rows."""
    if G == 1:
        return [0, S]
    ones = list(range(1, min(G, 3)))
    rest = np.random.default_rng(seed + G).choice(np.arange(len(ones) + 1, S), G - 1 - len(ones), replace=False)
    return [0] + ones + sorted(int(v) for v in rest) + [S]


def _wslabs(w, devices, bounds=None):
    """S x D host weights -> contiguous row slabs on `devices`."""
    from smart_crossover import device as dev
    S, D = w.shape
    sl = dev.CostSlabs(S, D, devices, bounds, pad_ld=False)
    for g in range(len(devices)):
        r0 = sl.row0[g]
        sl.t[g].copy_(torch.from_numpy(np.ascontiguousarray(w[r0:r0 + sl.rows[g]])))
    sl.sync()
    return sl


def _ids(t, kruskal):
    a = t.cpu().numpy()
    return a.view(np.uint32).astype(np.int64) if kruskal else a


def _check_head(w, head, T, kruskal):
    """`head` is the first m >= T arcs of the order, and the next arc is strictly lighter (whole tie runs)."""
    flat = w.ravel()
    ref = np.argsort(-flat, kind="stable") if kruskal else np.argsort(flat, kind="stable")[::-1]
    got = _ids(head, kruskal)
    m = got.size
    assert m >= min(T, flat.size)
    assert np.array_equal(got, ref[:m])
    if m < flat.size:
        assert flat[ref[m]] < flat[ref[m - 1]]


_SHAPES = [(257, 131), (1500, 1501)]            # n below and above 2^21


@pytest.mark.gpu
@pytest.mark.parametrize("G,uneven", [(1, False)] + [(G, u) for G in (2, 3, 5, 8) for u in (False, True)])
@pytest.mark.parametrize("shape", _SHAPES)
def test_head_matches_stable_argsort(G, uneven, shape):
    _need_cuda()
    from smart_crossover import device as dev
    S, D = shape
    rng = np.random.default_rng(S + G)
    w = rng.random((S, D)) ** 3
    sl = _wslabs(w, [torch.cuda.current_device()] * G, _uneven(S, G) if uneven else None)
    T = 16 * (S + D)
    for kruskal in (True, False):
        head = dev.order_head_sharded(sl, T, queue=not kruskal)
        _check_head(w, head, T, kruskal)
    # level-0 histograms taken beforehand (as sx_score_ot takes them while scoring) give the same head
    from smart_crossover._native import lib
    hists = [torch.zeros(4096, dtype=torch.int32, device=t.device) for t in sl.t]
    for t, h in zip(sl.t, hists):
        with torch.cuda.device(t.device):
            assert lib.sx_hist12_f64(dev._ptr(t), t.numel(), dev._ptr(h), dev._stream()) == 0
    _check_head(w, dev.order_head_sharded(sl, T, hists=hists), T, True)


@pytest.mark.gpu
@pytest.mark.parametrize("G,T_cap", [(1, 2000), (3, 2000), (8, 2000), (5, None)])
def test_head_with_a_crowded_threshold_bin(G, T_cap):
    """Integer scores: half the arcs share the threshold's level-0 bin.  A shard whose part of it overflows its
    boundary list (4 T_cap arcs) histograms and filters all its weights; 1-row shards keep to their lists."""
    _need_cuda()
    from smart_crossover import device as dev
    S, D = 1500, 1501
    w = np.random.default_rng(7 + G).integers(0, 1 << 20, size=(S, D)).astype(np.float64)
    sl = _wslabs(w, [torch.cuda.current_device()] * G, _uneven(S, G))
    for kruskal in (True, False):
        head = dev.order_head_sharded(sl, 1000, T_cap, queue=not kruskal)
        assert head is not None
        _check_head(w, head, 1000, kruskal)


@pytest.mark.gpu
@pytest.mark.parametrize("G", [1, 3])
def test_tie_run_longer_than_T_cap(G):
    """A tie run across the threshold longer than T_cap: the entry point returns None (-1), and the head of
    `ShardedScores` repeats with a larger capacity."""
    _need_cuda()
    from smart_crossover import device as dev
    from smart_crossover.network_methods.net_manager import ShardedScores
    S, D = 257, 131
    w = np.ones((S, D))
    w[5, :7] = 2.0
    sl = _wslabs(w, [torch.cuda.current_device()] * G, _uneven(S, G))
    assert dev.order_head_sharded(sl, 100, 1000) is None
    assert dev.order_head_sharded(sl, 100, 1000, queue=True) is None
    sc = ShardedScores(sl)
    for kruskal in (True, False):
        _check_head(w, sc.head(100, kruskal, T_cap=1000), 100, kruskal)


@pytest.mark.gpu
@pytest.mark.parametrize("G", [1, 5])
def test_signed_zeros_tie(G):
    """-0.0 == +0.0: both zeros form one tie run, ordered by id (NumPy order)."""
    _need_cuda()
    from smart_crossover import device as dev
    S, D = 257, 131
    rng = np.random.default_rng(11)
    w = np.where(rng.random((S, D)) < 0.5, 0.0, -0.0)
    w[rng.random((S, D)) < 0.01] = 1.5
    sl = _wslabs(w, [torch.cuda.current_device()] * G, _uneven(S, G))
    T = int((w > 0).sum()) + 10
    for kruskal in (True, False):
        _check_head(w, dev.order_head_sharded(sl, T, S * D, queue=not kruskal), T, kruskal)


@pytest.mark.gpu
def test_nan_scores_raise():
    _need_cuda()
    from smart_crossover.network_methods.net_manager import NAN_WEIGHTS_MSG, ShardedScores
    w = np.random.default_rng(3).random((40, 30))
    w[33, 4] = np.nan
    sc = ShardedScores(_wslabs(w, [torch.cuda.current_device()] * 2, [0, 30, 40]))
    for kruskal in (True, False):
        with pytest.raises(ValueError, match="NaN"):
            sc.head(10, kruskal)
    assert "NaN" in NAN_WEIGHTS_MSG


def _sharded_problem(s, d, M, x, devices, bounds=None):
    """Device-resident cost slabs, the flow as slabs like them, and a manager over them."""
    from smart_crossover import device as dev
    from smart_crossover.formats import OptTransport
    from smart_crossover.network_methods.net_manager import DeviceResidentCost, OTManager
    slabs = dev.CostSlabs.from_host(M, devices, row_bounds=bounds)
    flow = dev.CostSlabs.from_host(x, like=slabs)
    ot = OptTransport(s.copy(), d.copy(), DeviceResidentCost(slabs))
    return OTManager(ot), flow, ot


@pytest.mark.gpu
@pytest.mark.parametrize("G", [1, 3])
def test_tree_784_matches_host_tree_and_push_count(G):
    _need_cuda()
    from golden_util import c2_inputs
    from smart_crossover.network_methods.tree_BI import max_weight_spanning_tree, tree_basis_identify
    s, d, M, x = c2_inputs()
    small = Fixture("ot_c2_784_small")
    mgr, flow, ot = _sharded_problem(s, d, M, x, [torch.cuda.current_device()] * G, _uneven(784, G))
    queue, scores = mgr.get_sorted_flows(flow)
    assert len(queue) == scores.shape[0] == 784 * 784
    with pytest.raises(TypeError):
        np.asarray(scores)                                   # no host copy
    assert np.array_equal(max_weight_spanning_tree(ot, scores), small.out["tree"])
    basis, it = tree_basis_identify(mgr, scores)
    assert it == int(small.out["push_iter"]) == 934
    assert np.array_equal(np.flatnonzero(basis.vbasis == 0), small.out["basic_tree"])
    # host weights on the same manager take the host route even though the sharded scores are kept
    assert tree_basis_identify(mgr, orc.ot_flow_scores(x, s, d))[1] == 934
    ids = np.array([0, 5, 784 * 784 - 1, 123457])
    assert scores.take(ids).tobytes() == orc.ot_flow_scores(x, s, d)[ids].tobytes()


@pytest.mark.gpu
def test_tree_3000_matches_host_device_tree():
    _need_cuda()
    from smart_crossover.formats import OptTransport
    from smart_crossover.network_methods.net_manager import OTManager
    from smart_crossover.network_methods.tree_BI import _device_tree, tree_basis_identify
    S = D = 3000
    s, d, M = cases.ot_points(S, D, 3000)
    x = cases.interior_flow(s, d, M, 3000, 0.33)
    host_mgr = OTManager(OptTransport(s, d, M))
    _, host_scores = host_mgr.get_sorted_flows(x)
    host_tree, host_nt = _device_tree(host_mgr.ot, host_scores)
    host_basis, host_it = tree_basis_identify(host_mgr, host_scores)
    mgr, flow, ot = _sharded_problem(s, d, M, x, [torch.cuda.current_device()] * 4, _uneven(S, 4))
    _, scores = mgr.get_sorted_flows(flow)
    tree, nt = _device_tree(ot, scores, mgr._sorted)
    assert nt == host_nt == S + D - 1
    assert np.array_equal(tree[:nt].cpu().numpy(), host_tree[:host_nt].cpu().numpy())
    basis, it = tree_basis_identify(mgr, scores)
    assert it == host_it and np.array_equal(basis.vbasis, host_basis.vbasis)


def _cg_slices(m, n):
    """The slices `column_generation` takes of the queue (chunk doubling from int(1.2 m) when n / m <= 1000)."""
    left, target = 0, int(10 * m) if n / m > 1000 else int(1.2 * m)
    while left < n:
        right = min(target, n)
        yield left, right
        left, target = right, 2 * target


@pytest.mark.gpu
@pytest.mark.parametrize("G", [1, 5])
def test_queue_slices_match_host_queue(G):
    _need_cuda()
    from golden_util import c2_inputs
    from smart_crossover.formats import OptTransport
    from smart_crossover.network_methods.net_manager import OTManager
    s, d, M, x = c2_inputs()
    host_queue, _ = OTManager(OptTransport(s, d, M)).get_sorted_flows(x)
    mgr, flow, _ = _sharded_problem(s, d, M, x, [torch.cuda.current_device()] * G, _uneven(784, G))
    queue, _ = mgr.get_sorted_flows(flow)
    n = len(queue)
    for a, b in _cg_slices(784 + 784, n):
        got = queue[a:b]
        assert got.dtype == np.int64 and np.array_equal(got, host_queue[a:b])


@pytest.mark.gpu
def test_flow_slabs_must_match_the_cost_slabs():
    _need_cuda()
    from smart_crossover import device as dev
    s, d, M = cases.ot_points(60, 50, 5)
    cur = torch.cuda.current_device()
    mgr, _, _ = _sharded_problem(s, d, M, np.full(60 * 50, 1e-3), [cur, cur], [0, 20, 60])
    other = dev.CostSlabs.from_host(np.full((60, 50), 1e-3), like=dev.CostSlabs(60, 50, [cur, cur], [0, 30, 60]))
    with pytest.raises(ValueError, match="row bounds"):
        mgr.get_sorted_flows(other)
    # a manager over a host matrix refuses flow slabs without uploading the matrix first
    from smart_crossover.formats import OptTransport
    from smart_crossover.network_methods.net_manager import OTManager
    host = OTManager(OptTransport(s, d, M))
    with pytest.raises(ValueError, match="row bounds"):
        host.get_sorted_flows(other)
    assert host._slabs is None


@pytest.mark.gpu
@pytest.mark.parametrize("G", [1, 3])
def test_sinkhorn_flow_slabs_equal_the_host_plan_rows(G):
    _need_cuda()
    from smart_crossover import device as dev
    from smart_crossover.warm_start import sinkhorn
    S, D = 257, 131
    s, d, M = cases.ot_points(S, D, 21)
    slabs = dev.CostSlabs.from_host(M, [torch.cuda.current_device()] * G, row_bounds=_uneven(S, G))
    plan = sinkhorn(s, d, slabs, 0.05, numItermax=200, stopThr=0.0)
    X, info = sinkhorn(s, d, slabs, 0.05, numItermax=200, stopThr=0.0, log=True, as_slabs=True)
    assert info["niter"] == 200 and X.same_shards(dev.CostSlabs.from_host(plan, like=slabs))
    for g in range(G):
        r0 = slabs.row0[g]
        assert X.t[g].cpu().numpy().tobytes() == plan[r0:r0 + slabs.rows[g]].tobytes()


def _e2e_784(devices):
    from golden_util import c2_inputs
    from smart_crossover.network_methods.algorithms import network_crossover
    from smart_crossover.solver_caller.caller import SolverSettings
    s, d, M, x = c2_inputs()
    fx = Fixture("e2e_c2_784")
    _, flow, ot = _sharded_problem(s, d, M, x, devices)
    out = network_crossover(x=flow, ot=ot, method="tnet", solver="HGS", solver_settings=SolverSettings(log_console=0))
    ref = float(fx.out["tnet_obj"])
    assert abs(out.obj_val - ref) <= 1e-9 * abs(ref)
    assert out.iter_count == int(fx.out["tnet_iters"])
    assert np.array_equal(np.flatnonzero(out.basis.vbasis == 0), fx.out["tnet_basic"])


@pytest.mark.gpu
def test_network_crossover_tnet_on_device_resident_784():
    _need_cuda()
    _e2e_784([torch.cuda.current_device()])


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, "all"])
def test_distinct_devices_match_the_emulation(n):
    """Head (both modes), tree and queue from shards on distinct GPUs == the same bounds on one GPU, byte for byte;
    and TNET end to end on the 784^2 golden with the slabs on those GPUs."""
    n_vis = _n_gpus()
    if n_vis < 2:
        pytest.skip("needs at least 2 GPUs")
    from golden_util import c2_inputs
    from smart_crossover import device as dev
    from smart_crossover.network_methods.tree_BI import _device_tree
    G = n_vis if n == "all" else 2
    S, D = 1500, 1501
    w = np.random.default_rng(G).random((S, D))
    bounds = _uneven(S, G)
    heads = []
    for devices in ([0] * G, list(range(G))):
        sl = _wslabs(w, devices, bounds)
        heads.append([dev.order_head_sharded(sl, 16 * (S + D), queue=q).cpu().numpy().tobytes() for q in (0, 1)])
    assert heads[0] == heads[1]
    s, d, M, x = c2_inputs()
    runs = []
    for devices in ([0] * G, list(range(G))):
        mgr, flow, ot = _sharded_problem(s, d, M, x, devices, _uneven(784, G))
        queue, scores = mgr.get_sorted_flows(flow)
        tree, nt = _device_tree(ot, scores, mgr._sorted)
        runs.append((tree[:nt].cpu().numpy().tobytes(), [queue[a:b].tobytes() for a, b in _cg_slices(1568, len(queue))]))
    assert runs[0] == runs[1]
    _e2e_784(list(range(G)))

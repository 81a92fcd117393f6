"""Parity of the CUDA path (through the C ABI of libsxcross) against the CPU oracle and the
golden vectors produced by the reference.  Run on a B200: `pytest -m gpu`.

Bars (BASELINE.json north_star): sorted arc order, tree arc set and selected column set
bit-exact; reduced costs bitwise for the same duals; potentials within 1e-9 relative.
"""
import numpy as np
import pytest

import cases
from golden_util import MCF_FULL, OT_FULL, Fixture, c2_inputs, digests, mcf_mid_inputs
from oracle import network_oracle as orc

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
RTOL = 1e-9


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from smart_crossover import device
    return device


@pytest.fixture(params=["fused", "separate"])
def fused_mode(request, dev):
    """Dense pricing passes through the fused kernel (price + select in one launch) or the separate ones."""
    old = dev.FUSED_DEFAULT
    dev.FUSED_DEFAULT = request.param == "fused"
    yield request.param
    dev.FUSED_DEFAULT = old


def cu(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda()


def price_in_one_fused_launch(dev, pr, M, y, K):
    """price_dense_ot through the fused pricer `pr`; the pass must be one launch of the fused kernel."""
    assert pr.fused
    before = pr.launches
    res = dev.price_dense_ot(cu(M), cu(y), K=K, pricer=pr)
    assert pr.launches == before + 1
    return res


def u32(t):
    """uint32 bit patterns stored in an int32 tensor -> int64 numpy."""
    return t.cpu().numpy().view(np.uint32).astype(np.int64)


def sort_pipeline(dev, key_t):
    order, skey = dev.argsort_f64(key_t)
    queue = dev.queue_from_order(order)
    korder = dev.kruskal_order(skey, order)
    return order, skey, queue, korder


def test_kruskal_order_head_is_the_head_of_the_flipped_order(dev):
    """sx_kruskal_order_head cuts whole tie runs from the end of the ascending sort: same arcs, same order
    as the first entries of the full Kruskal order; too long a run at the cut is reported."""
    rng = np.random.default_rng(5)
    for n, T, kind in [(100003, 1000, "random"), (100003, 5000, "ties"), (4096 * 3 + 1, 4097, "ties"),
                       (777, 777, "random"), (50000, 49999, "ties"), (10, 3, "random")]:
        key = rng.random(n)
        if kind == "ties":
            key = np.round(key * 300) / 300                          # runs of ~n / 300 equal keys
        order, skey, queue, korder = sort_pipeline(dev, cu(key))
        full = u32(korder)
        head = dev.kruskal_order_head(skey, order, T, T_cap=n)
        assert head is not None
        head = u32(head)
        assert T <= head.size <= n
        assert np.array_equal(head, full[:head.size])
        if head.size < n:                                            # the cut is at a run boundary
            assert key[full[head.size]] < key[head[-1]]
    key = np.zeros(5000)
    key[:10] = 1.0
    order, skey = dev.argsort_f64(cu(key))
    assert np.array_equal(u32(dev.kruskal_order_head(skey, order, 5, T_cap=20)), np.arange(10))
    assert dev.kruskal_order_head(skey, order, 11, T_cap=20) is None  # the zero run has 4990 arcs


# ---- K1a + K1c ------------------------------------------------------------------------------
def test_ot_scores_special_values_bitwise(dev):
    """K1a against NumPy on the awkward inputs: negative / zero / -0.0 / inf / NaN flows, zero, negative,
    infinite and NaN marginals, denormals, and 2e5 random positive triples (the one-division fast path
    must give the same bits as max(x / s, x / d))."""
    rng = np.random.default_rng(0)
    special = np.array([0.0, -0.0, 1.0, -1.0, 3.3e-310, 1e-300, 1e300, np.inf, -np.inf, np.nan, 0.1, 7.0])
    S = D = special.size
    s = special.copy()
    d = special[::-1].copy()
    X = np.tile(special, (S, 1)).T.copy()                      # x varies along rows, d along columns
    X2 = rng.permuted(np.tile(special, (S, 1)), axis=1)
    for xs in (X, X2):
        with np.errstate(all="ignore"):
            ref = np.maximum(xs / s[:, None], xs / d[None, :]).ravel()
        got = dev.score_ot(cu(xs.ravel()), cu(s), cu(d)).cpu().numpy()
        assert np.array_equal(np.isnan(got), np.isnan(ref))
        ok = ~np.isnan(ref)
        assert got[ok].tobytes() == ref[ok].tobytes()
    S, D = 400, 500
    s = 10.0 ** rng.uniform(-8, 3, S)
    d = 10.0 ** rng.uniform(-8, 3, D)
    x = 10.0 ** rng.uniform(-12, 2, S * D)
    x[rng.random(x.size) < 0.05] = 0.0
    ref = np.maximum(x.reshape(S, D) / s[:, None], x.reshape(S, D) / d[None, :]).ravel()
    assert dev.score_ot(cu(x), cu(s), cu(d)).cpu().numpy().tobytes() == ref.tobytes()


@pytest.mark.parametrize("name", OT_FULL + ["ot_zero_3x3"])
def test_ot_scores_and_orders_golden(dev, name):
    fx = Fixture(name)
    s, d, x = fx.inp["s"], fx.inp["d"], fx.inp["x"]
    F = dev.score_ot(cu(x), cu(s), cu(d))
    assert F.cpu().numpy().tobytes() == fx.out["scores"].tobytes()
    order, skey, queue, korder = sort_pipeline(dev, F)
    assert np.array_equal(queue.cpu().numpy(), fx.out["queue"])
    assert np.array_equal(u32(korder), orc.kruskal_order(fx.out["scores"]))
    assert skey.cpu().numpy().tobytes() == np.sort(fx.out["scores"], kind="stable").tobytes()


def test_c2_784_scores_queue_tree_potentials(dev):
    s, d, M, x = c2_inputs()
    dg = digests()["ot_c2_784"]["digests"]
    small = Fixture("ot_c2_784_small").out
    S, D = M.shape
    F = dev.score_ot(cu(x), cu(s), cu(d))
    assert cases.digest(F.cpu().numpy()) == dg["scores"]
    order, skey, queue, korder = sort_pipeline(dev, F)
    assert cases.digest(queue.cpu().numpy()) == dg["queue"]
    tree, n_tree = dev.kruskal(korder, S + D, S=S, D=D)
    nt = int(n_tree.item())
    assert nt == S + D - 1
    assert np.array_equal(tree[:nt].cpu().numpy(), small["tree"])
    y = dev.tree_potentials(tree, nt, S + D, cu(M), S + D - 1, S=S, D=D)
    np.testing.assert_allclose(y.cpu().numpy(), small["y_tree"], rtol=RTOL, atol=RTOL * M.max())
    # pricing against the stored perturbed duals: digest of the full rc vector, count, min, top-k
    res = dev.price_dense_ot(cu(M), cu(small["y_pert"]), K=256, want_rc=True)
    assert cases.digest(res.rc.cpu().numpy()) == dg["rc_pert"]
    assert res.n_violating == int(small["count_pert"])
    assert res.min_rc == float(small["min_rc_pert"])
    assert np.array_equal(res.topk_id, small["topk_ids_pert"])


@pytest.fixture(params=["one launch", "launch per pass"])
def sort_mode(request):
    """Mid-size sorts (8 K < n <= ~1.2 M keys) run every pass in one cooperative launch; the other parameter
    forces the upsweep / scan / downsweep launches that larger inputs use."""
    from smart_crossover._native import lib
    assert lib.sx_sort_set_tuning(1 if request.param == "one launch" else 0) == 0
    yield request.param
    assert lib.sx_sort_set_tuning(1) == 0 and lib.sx_sort_set_tuning(2) == 0


@pytest.mark.parametrize("n", [1, 2, 31, 4095, 4096, 4097, 8192, 8193, 70001, 614656, 1 << 20, 1212416, 1212417])
def test_argsort_edge_sizes_and_special_values(dev, sort_mode, n):
    rng = np.random.default_rng(n)
    key = rng.integers(-3, 4, size=n).astype(np.float64) * rng.choice([0.5, 1.0, 1e-300], size=n)
    if n > 8:
        key[::7] = 0.0
        key[3::11] = -0.0
        key[5::13] = np.inf
        key[6::17] = -np.inf
        key[2::19] = np.nan
    order, skey, queue, korder = sort_pipeline(dev, cu(key))
    ref = np.argsort(key, kind="stable")
    assert np.array_equal(u32(order), ref)
    assert np.array_equal(queue.cpu().numpy(), ref[::-1])
    got = skey.cpu().numpy()
    assert np.array_equal(np.isnan(got), np.isnan(key[ref]))
    assert np.array_equal(got[~np.isnan(got)], key[ref][~np.isnan(got)])
    if not np.isnan(key).any():
        assert np.array_equal(u32(korder), orc.kruskal_order(key))


@pytest.mark.parametrize("n,bits", [(3134, 11), (8192, 13), (20000, 20), (300000, 33), (1 << 20, 63), (100, 63)])
def test_argsort_u64_partial_key_bits(dev, sort_mode, n, bits):
    """sx_argsort_u64 looks at ceil(bits / 8) low bytes only (ties among them by index), on every size path."""
    import ctypes
    from smart_crossover._native import check, lib
    rng = np.random.default_rng(bits)
    key = rng.integers(0, 1 << min(bits, 62), size=n, dtype=np.int64).astype(np.uint64)
    key[::5] |= np.uint64(1) << np.uint64(63)                     # bits above the sorted range must be ignored ...
    passes = max(2, (bits + 7) // 8)
    masked = key & np.uint64((1 << (8 * passes)) - 1 if passes < 8 else 0xFFFFFFFFFFFFFFFF)
    ref = np.argsort(masked, kind="stable")
    kt = torch.from_numpy(key.view(np.int64)).cuda()
    order = torch.empty(n, dtype=torch.int32, device="cuda")
    skey = torch.empty(n, dtype=torch.int64, device="cuda")
    ws = torch.empty(lib.sx_argsort_workspace_bytes(n), dtype=torch.uint8, device="cuda")
    check(lib.sx_argsort_u64(dev._ptr(kt), n, bits, dev._ptr(order), dev._ptr(skey), dev._ptr(ws), ws.numel(),
                             dev._stream()), "sx_argsort_u64")
    assert np.array_equal(u32(order), ref)
    assert np.array_equal(skey.cpu().numpy().view(np.uint64), key[ref])           # ... but travel with the key


def test_kruskal_order_long_runs(dev):
    """Tie runs longer than a thread block and crossing block boundaries."""
    n = 50000
    key = np.repeat(np.array([3.0, 1.0, 2.0, 2.0, 0.5]), n // 5)
    key[12345] = 7.0
    order, skey, queue, korder = sort_pipeline(dev, cu(key))
    assert np.array_equal(u32(korder), orc.kruskal_order(key))
    key = np.zeros(20000)
    order, skey, queue, korder = sort_pipeline(dev, cu(key))
    assert np.array_equal(u32(korder), np.arange(20000))


# ---- K2 / K3 -----------------------------------------------------------------------------------
@pytest.mark.parametrize("name", OT_FULL + ["ot_zero_3x3"])
def test_tree_and_potentials_golden(dev, name):
    fx = Fixture(name)
    M = fx.inp["M"]
    S, D = M.shape
    F = cu(fx.out["scores"])
    order, skey, queue, korder = sort_pipeline(dev, F)
    tree, n_tree = dev.kruskal(korder, S + D, S=S, D=D)
    nt = int(n_tree.item())
    got = tree[:nt].cpu().numpy()
    assert nt == S + D - 1
    # the reference drops zero-weight tree arcs (SURVEY.md H2); the host mirror applies the same filter
    assert np.array_equal(got[fx.out["scores"][got] != 0], fx.out["tree"])
    assert np.array_equal(got, orc.max_weight_spanning_tree(fx.out["scores"], S, D, drop_zero_weight=False))
    if "y_tree" in fx.out:
        y = dev.tree_potentials(tree, nt, S + D, cu(M), S + D - 1, S=S, D=D)
        np.testing.assert_allclose(y.cpu().numpy(), fx.out["y_tree"], rtol=RTOL, atol=RTOL * np.abs(M).max())


@pytest.mark.parametrize("N,E,seed", [(50, 49, 1), (300, 2000, 2), (5000, 40000, 3), (20000, 25000, 4)])
def test_kruskal_general_graph(dev, N, E, seed):
    """Arc-list endpoints (C3 shape), possibly disconnected: forest equals sequential Kruskal."""
    rng = np.random.default_rng(seed)
    tail = rng.integers(0, N, size=E)
    head = (tail + 1 + rng.integers(0, N - 1, size=E)) % N
    w = rng.integers(1, 50, size=E).astype(np.float64)       # heavy ties
    order, skey, queue, korder = sort_pipeline(dev, cu(w))
    tree, n_tree = dev.kruskal(korder, N, tail=cu(tail, torch.int32), head=cu(head, torch.int32))
    nt = int(n_tree.item())
    ref = orc.spanning_forest(orc.kruskal_order(w), N, tail=tail, head=head)
    assert nt == ref.size
    assert np.array_equal(tree[:nt].cpu().numpy(), ref)
    if nt == N - 1:
        cost = rng.integers(1, 100, size=E).astype(np.float64)
        y = dev.tree_potentials(tree, nt, N, cu(cost), N - 1, tail=cu(tail, torch.int32),
                                head=cu(head, torch.int32), plus=1)
        yr = orc.tree_potentials(tail[ref], head[ref], cost[ref], N, N - 1)
        np.testing.assert_allclose(y.cpu().numpy(), yr, rtol=RTOL, atol=RTOL * 100)


def test_tree_potentials_rejects_non_spanning(dev):
    from smart_crossover._native import SxError, SX_ERR_NOT_SPANNING
    S = D = 4
    M = np.arange(16, dtype=np.float64).reshape(4, 4)
    # 7 arcs containing a 4-cycle (0,0),(0,1),(1,0),(1,1): not a tree
    tree = np.array([0, 1, 4, 5, 10, 11, 15], dtype=np.int64)
    with pytest.raises(SxError) as ei:
        dev.tree_potentials(cu(tree), 7, S + D, cu(M), S + D - 1, S=S, D=D)
    assert ei.value.code == SX_ERR_NOT_SPANNING
    with pytest.raises(SxError):
        dev.tree_potentials(cu(tree[:5]), 5, S + D, cu(M), S + D - 1, S=S, D=D)


@pytest.mark.parametrize("S,D,T,kind", [(300, 400, 5000, "interior"), (64, 5000, 20000, "interior"),
                                        (500, 500, 16000, "ties"), (257, 129, 1, "interior"),
                                        (200, 300, 60000, "interior"), (128, 128, 3000, "zeros")])
def test_kruskal_prefix_is_the_head_of_the_full_order(dev, S, D, T, kind):
    """sx_kruskal_prefix == the first entries of argsort + kruskal_order, for generic weights, for
    product weights with massive ties (SURVEY.md H1) and with exact zeros."""
    s, d, M = cases.ot_points(S, D, 900 + S)
    if kind == "ties":
        x = np.outer(s, d).ravel()                                   # every score ties along rows / columns
    else:
        x = cases.interior_flow(s, d, M, 900 + S, 0.33)
        if kind == "zeros":
            x[np.random.default_rng(1).random(x.size) < 0.7] = 0.0
    F = orc.ot_flow_scores(x, s, d)
    order, skey, queue, korder = sort_pipeline(dev, cu(F))
    full = korder.cpu().numpy().view(np.uint32)
    head = dev.kruskal_prefix(cu(F), T, T_cap=S * D)
    assert head is not None
    head = head.cpu().numpy().view(np.uint32)
    assert min(T, S * D) <= head.size <= S * D
    assert np.array_equal(head, full[:head.size])
    # everything left out is strictly lighter than the lightest arc kept (to 24 bits of the key)
    if head.size < S * D:
        assert F[full[head.size]] < F[head[-1]]
    # capacity too small for the ties at the threshold: the caller is told to sort everything
    if kind == "ties":
        assert dev.kruskal_prefix(cu(F), 10, T_cap=12) is None
    # the level-0 histogram taken by the score kernel (vector path when D is even) gives the same head
    Ft, hist = dev.score_ot(cu(x), cu(s), cu(d), want_hist=True)
    assert Ft.cpu().numpy().tobytes() == F.tobytes()
    keys = F.view(np.uint64) | np.uint64(1 << 63)                     # scores are >= 0: image = bits | sign
    ref_hist = np.bincount((keys >> np.uint64(52)).astype(np.int64), minlength=4096)
    assert np.array_equal(hist.cpu().numpy().astype(np.int64), ref_hist)
    head2 = dev.kruskal_prefix(Ft, T, T_cap=S * D, hist=hist)
    assert np.array_equal(head2.cpu().numpy().view(np.uint32), head)


@pytest.mark.parametrize("n,T,T_cap", [(1 << 20, 1000, 4096), (300001, 2000, 3000), (1 << 20, 1000, 1 << 20)])
def test_kruskal_prefix_crowded_threshold_bin(dev, n, T, T_cap):
    """All weights share one exponent (one level-0 bin): with a small T_cap the boundary list of the
    split pass overflows and the second level streams every weight again; with a large T_cap it is
    resolved from the list.  Either way the head equals the head of the full sort."""
    rng = np.random.default_rng(n + T)
    w = 1.0 + rng.random(n)
    w[rng.integers(0, n, 200)] = 1.9999                               # exact ties inside the head
    order, skey, queue, korder = sort_pipeline(dev, cu(w))
    full = korder.cpu().numpy().view(np.uint32)
    head = dev.kruskal_prefix(cu(w), T, T_cap=T_cap)
    assert head is not None
    head = head.cpu().numpy().view(np.uint32)
    assert T <= head.size <= T_cap
    assert np.array_equal(head, full[:head.size])
    assert w[full[head.size]] < w[head[-1]]


def test_tree_from_prefix_equals_tree_from_full_sort(dev):
    from smart_crossover.formats import OptTransport
    from smart_crossover.network_methods import tree_BI
    from smart_crossover.network_methods.net_manager import OTManager
    S, D = 400, 700
    s, d, M = cases.ot_points(S, D, 31)
    x = cases.interior_flow(s, d, M, 31, 0.33)
    F = orc.ot_flow_scores(x, s, d)
    ot = OptTransport(s, d, M)
    tree_ref = orc.max_weight_spanning_tree(F, S, D)
    assert not tree_BI.use_prefix_path(S * D, S + D)                  # small instance: full argsort by default
    assert np.array_equal(tree_BI.max_weight_spanning_tree(ot, F), tree_ref)
    old, old_min = tree_BI.PREFIX_FACTOR, tree_BI.PREFIX_MIN_ARCS
    try:
        tree_BI.PREFIX_MIN_ARCS = 0                                   # force the path large instances take
        assert tree_BI.use_prefix_path(S * D, S + D)
        assert np.array_equal(tree_BI.max_weight_spanning_tree(ot, F), tree_ref)
        mgr = OTManager(ot)
        q, F2 = mgr.get_sorted_flows(x)                               # full sort exists: its head is reused
        assert np.array_equal(tree_BI.max_weight_spanning_tree(ot, F2, _sorted=mgr._sorted), tree_ref)
        tree_BI.PREFIX_FACTOR = 1                                     # head too short: falls back, same tree
        assert np.array_equal(tree_BI.max_weight_spanning_tree(ot, F), tree_ref)
        assert np.array_equal(tree_BI.max_weight_spanning_tree(ot, F2, _sorted=mgr._sorted), tree_ref)
    finally:
        tree_BI.PREFIX_FACTOR, tree_BI.PREFIX_MIN_ARCS = old, old_min


@pytest.mark.parametrize("name", OT_FULL)
def test_tree_flows_golden(dev, name):
    """Tree primal flows (SuperLU in the reference, tree_BI.py:74-76) from the Euler tour, and the push
    phase driven by them: same basis and push count as the reference."""
    from smart_crossover.formats import OptTransport
    from smart_crossover.network_methods.net_manager import OTManager
    from smart_crossover.network_methods.tree_BI import push_tree_to_bfs, tree_flows
    fx = Fixture(name)
    s, d, M = fx.inp["s"], fx.inp["d"], fx.inp["M"]
    ot = OptTransport(s, d, M)
    flows = tree_flows(ot, fx.out["tree"])
    np.testing.assert_allclose(flows, fx.out["tree_flows"], rtol=1e-9, atol=1e-12 * max(s.max(), d.max()))
    vbasis, push_iter = push_tree_to_bfs(OTManager(ot), fx.out["tree"])
    assert push_iter == int(fx.out["push_iter"])
    assert np.array_equal(vbasis.astype(np.int64), fx.out["vbasis_tree"])


def test_tree_flows_are_exact_subtree_sums(dev):
    """Integer supplies: every subtree sum is exactly representable, so the flows must be exact,
    and A[:, tree] @ flows == b on every node but the root (conservation)."""
    S, D = 300, 500
    rng = np.random.default_rng(8)
    s = rng.integers(1, 1000, S).astype(np.float64)
    d = rng.integers(1, 1000, D).astype(np.float64)
    d[-1] += s.sum() - d.sum()
    M = rng.random((S, D))
    F = rng.random(S * D)
    tree = orc.max_weight_spanning_tree(F, S, D)
    b = np.hstack([-s, d])
    flows = dev.tree_flows(cu(tree), tree.size, S + D, cu(b), S + D - 1, S=S, D=D).cpu().numpy()
    assert np.array_equal(flows, np.round(flows))
    bal = np.zeros(S + D)
    np.add.at(bal, tree // D, -flows)
    np.add.at(bal, S + tree % D, flows)
    assert np.array_equal(bal[:-1], b[:-1])
    # arc-list form, min2mcf sign convention (+1 at the tail)
    tail = (S + tree % D).astype(np.int32)
    head = (tree // D).astype(np.int32)
    from smart_crossover._native import SX_PLUS_IS_TAIL
    ids = np.arange(tree.size, dtype=np.int64)
    f2 = dev.tree_flows(cu(ids), tree.size, S + D, cu(b), S + D - 1, tail=cu(tail), head=cu(head),
                        plus=SX_PLUS_IS_TAIL).cpu().numpy()
    assert np.array_equal(f2, flows)


# ---- K4 ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", OT_FULL)
@pytest.mark.parametrize("variant", [-1, 0, 1, 2])
def test_price_dense_golden(dev, name, variant):
    fx = Fixture(name)
    M = fx.inp["M"]
    S, D = M.shape
    if variant in (0, 1) and D % 2:
        from smart_crossover._native import SxError
        with pytest.raises(SxError):
            dev.price_dense_ot(cu(M), cu(fx.out["y_pert"]), K=8, variant=variant)
        return
    for tag in ("tree", "pert"):
        res = dev.price_dense_ot(cu(M), cu(fx.out["y_" + tag]), K=64, want_rc=True, variant=variant)
        rc_ref = fx.out["rc_" + tag]
        assert res.rc.cpu().numpy().tobytes() == rc_ref.tobytes()      # bitwise (SURVEY.md H4)
        cnt, mn, ids, vals = orc.price_summary(rc_ref, K=64)
        assert res.n_violating == cnt and res.min_rc == mn
        assert res.optimal == bool(fx.out["optimal_" + tag])
        assert np.array_equal(res.topk_id, ids) and np.array_equal(res.topk_rc, vals)


@pytest.mark.parametrize("S,D,K,noise", [(1, 1, 4, 0.5), (3, 700, 16, 0.3), (257, 513, 1024, 0.2),
                                         (1000, 1002, 5000, 0.05), (2049, 4100, 100, 0.01),
                                         (4096, 4096, 1024, 0.0)])
@pytest.mark.parametrize("variant", [-1, 1, 2])
def test_price_dense_random_shapes(dev, fused_mode, S, D, K, noise, variant):
    if variant == 1 and D % 2:
        pytest.skip("vector loads need an even leading dimension")
    s, d, M = cases.ot_points(S, D, 1000 + S)
    y = cases.planted_duals(M, S, noise)
    rc_ref = orc.reduced_costs_ot(M, y)
    cnt, mn, ids, vals = orc.price_summary(rc_ref, K=K)
    res = dev.price_dense_ot(cu(M), cu(y), K=K, want_rc=(S * D < 2_000_000), variant=variant)
    assert res.n_violating == cnt and res.min_rc == mn
    assert np.array_equal(res.topk_id, ids) and np.array_equal(res.topk_rc, vals)
    if res.rc is not None:
        assert res.rc.cpu().numpy().tobytes() == rc_ref.tobytes()
    if noise == 0.0:
        assert res.optimal


@pytest.mark.parametrize("variant", [-1, 1, 2])
@pytest.mark.parametrize("where", ["cost", "source dual", "sink dual"])
def test_price_nan_reduced_cost_is_not_optimal(dev, fused_mode, variant, where):
    """A NaN reduced cost: `np.all(rc >= -tol)` (net_manager.py:496) is False, `(rc < -tol).sum()` does not
    count it and NumPy's argsort puts it last.  The device pass must report the same three things."""
    S, D = 130, 514
    s, d, M = cases.ot_points(S, D, 77)
    y = cases.planted_duals(M, 77, 0.0)
    y[S:] -= 1e-3                                    # strictly dual feasible: no violator
    M = M.copy()
    if where == "cost":
        M[S - 1, D - 3] = np.nan
    elif where == "source dual":
        y[5] = np.nan
    else:
        y[S + 511] = np.nan
    rc_ref = orc.reduced_costs_ot(M, y)
    assert np.isnan(rc_ref).any() and not np.all(rc_ref >= -1e-6) and (rc_ref < -1e-6).sum() == 0
    res = dev.price_dense_ot(cu(M), cu(y), K=8, want_rc=True, variant=variant)
    assert res.rc.cpu().numpy().tobytes() == rc_ref.tobytes()
    assert res.n_violating == 0 and res.topk_id.size == 0
    assert res.has_nan and not res.optimal
    # with violators present the NaN still is not one of them
    y2 = cases.planted_duals(M, 78, 0.2)
    if where != "cost":
        y2[5 if where == "source dual" else S + 511] = np.nan
    rc2 = orc.reduced_costs_ot(M, y2)
    cnt, mn, ids, vals = orc.price_summary(rc2, K=64)
    res = dev.price_dense_ot(cu(M), cu(y2), K=64, variant=variant)
    assert res.n_violating == cnt and res.min_rc == np.nanmin(rc2) and res.has_nan and not res.optimal
    assert np.array_equal(res.topk_id, ids) and res.topk_rc.tobytes() == vals.tobytes()
    # arc-list pricing raises the same flag: rc = c - (y[plus] - y[minus]) with plus = sink, minus = source
    if variant == -1:
        minus = np.repeat(np.arange(S), D).astype(np.int32)
        plus = (S + np.tile(np.arange(D), S)).astype(np.int32)
        ra = dev.price_arcs(cu(M.ravel()), cu(plus), cu(minus), cu(y2), K=64)
        assert ra.n_violating == cnt and ra.has_nan and not ra.optimal and np.array_equal(ra.topk_id, ids)


def test_price_tied_reduced_costs_and_overflow(dev, fused_mode):
    """Integer costs and duals: massive rc ties (broken by arc id); candidate buffer smaller
    than the violator count forces the exact re-pricing path."""
    s, d, M = cases.ot_grid(12, 5)          # 144 x 144, integer costs
    rng = np.random.default_rng(5)
    y = rng.integers(-40, 40, size=288).astype(np.float64)
    rc_ref = orc.reduced_costs_ot(M, y)
    for K in (7, 512, 3000):
        cnt, mn, ids, vals = orc.price_summary(rc_ref, K=K)
        pr = dev.Pricer(torch.device("cuda"), K, cand_cap=100)
        res = dev.price_dense_ot(cu(M), cu(y), K=K, pricer=pr)
        assert cnt > 100 and pr.cap > 100                  # grew after SX_STATUS_CAND_OVERFLOW
        assert res.n_violating == cnt and np.array_equal(res.topk_id, ids) and np.array_equal(res.topk_rc, vals)


@pytest.mark.parametrize("frac,K", [(0.5, 64), (0.5, 1024), (0.9, 1), (0.02, 1024), (0.3, 4000)])
def test_price_many_violators_are_pruned(dev, fused_mode, frac, K):
    """A far-from-optimal y (10 % - 90 % of all arcs violate): the count stays exact, the candidate
    list stays short (running histogram bound) and the top-K is still exact."""
    S, D = 6000, 4096
    rng = np.random.default_rng(int(frac * 100) + K)
    M = rng.random((S, D))
    y = np.concatenate([np.zeros(S), np.full(D, frac)])            # rc = M - frac: `frac` of the arcs < 0
    y[:S] += rng.normal(0, 0.01, S)
    rc_ref = orc.reduced_costs_ot(M, y)
    cnt, mn, ids, vals = orc.price_summary(rc_ref, K=K)
    pr = dev.Pricer(torch.device("cuda"), K)
    res = dev.price_dense_ot(cu(M), cu(y), K=K, pricer=pr)
    assert res.n_violating == cnt and res.min_rc == mn and cnt > 0.9 * frac * S * D
    assert np.array_equal(res.topk_id, ids) and np.array_equal(res.topk_rc, vals)
    n_cand = pr.n_candidates()
    assert 0 < n_cand < cnt // 4, f"pruning kept {n_cand} of {cnt} violators"
    assert pr.status == 0


def test_price_all_equal_reduced_costs(dev, fused_mode):
    """Every arc has the same reduced cost: no bound can prune and 60 000 candidates tie at the K-th
    value; the selection refines on the arc id (ids win ties)."""
    S, D, K = 300, 200, 100
    M = np.full((S, D), 2.0)
    y = np.concatenate([np.zeros(S), np.full(D, 3.0)])            # rc = -1 everywhere
    pr = dev.Pricer(torch.device("cuda"), K)
    if fused_mode == "fused":
        res = price_in_one_fused_launch(dev, pr, M, y, K)
    else:
        res = dev.price_dense_ot(cu(M), cu(y), K=K, pricer=pr)
    assert res.n_violating == S * D and res.min_rc == -1.0
    assert np.array_equal(res.topk_id, np.arange(K)) and np.all(res.topk_rc == -1.0)
    assert pr.status == 0


@pytest.mark.parametrize("K", [501, 1024])
def test_selection_refines_key_and_large_ids_within_the_level_bound(dev, K):
    """The boundary bin holds 100 000 exact ties at rank K plus a few thousand near-ties that differ from
    them only in low mantissa bits, and the arc ids straddle 2^62: the selection has to refine on the key
    first, then on the high and low bits of the id, and still finishes with the exact top K."""
    rng = np.random.default_rng(K)
    tie = -(1.0 + 2.0 ** -9 + 12345 * 2.0 ** -52)                 # middle of its 0.4 %-wide histogram bin
    rc = np.concatenate([
        -3.0 + rng.random(500),                                   # the 500 best arcs, in lower bins
        np.full(100_000, tie),                                    # rank K falls inside this tie
        tie + rng.integers(1, 12345, 3000) * 2.0 ** -52,          # same bin as the tie, above it in the low bits
        tie + rng.integers(1 << 30, 1 << 40, 3000) * 2.0 ** -52,  # same bin, higher key bits
        rng.random(2000)])                                        # not violating
    rc = rc[rng.permutation(rc.size)]
    id0 = 2 ** 62 - 50_000
    n_nodes = 64
    tail = rng.integers(0, n_nodes, rc.size).astype(np.int32)
    head = rng.integers(0, n_nodes, rc.size).astype(np.int32)
    y = np.zeros(n_nodes)                                         # rc = c - (0 - 0) = c exactly
    cnt, mn, ids, vals = orc.price_summary(rc, K=K)
    assert vals[499] < tie == vals[500] == vals[-1]                 # rank K lies inside the tie
    pr = dev.Pricer(torch.device("cuda"), K)
    pr.reset()
    pr.price_arcs(cu(rc), cu(tail), cu(head), None, cu(y), id0=id0)
    pr.select()
    res = pr.fetch()
    assert pr.status == 0 and res.n_violating == cnt
    assert np.array_equal(res.topk_id, ids + id0) and res.topk_rc.tobytes() == vals.tobytes()


def test_selection_flags_an_arc_priced_into_one_pass_many_times(dev):
    """A pass that prices the same arc 8 300 times leaves more copies of one (rc, id) than the selection can
    rank: the result is void, SX_STATUS_DUPLICATE_CANDIDATES is raised and `fetch` refuses it."""
    from smart_crossover import _native
    pr = dev.Pricer(torch.device("cuda"), 16)
    c, tail, head, y = cu(np.array([-1.0])), cu(np.array([0], np.int32)), cu(np.array([1], np.int32)), cu(np.zeros(2))
    pr.reset()
    for _ in range(8300):
        pr.price_arcs(c, tail, head, None, y)
    pr.select()
    with pytest.raises(ValueError):
        pr.fetch()
    assert pr.status & _native.SX_STATUS_DUPLICATE_CANDIDATES


def test_price_near_ties_at_the_kth_value(dev, fused_mode):
    """One tight arc per column shifted by the same delta (bench.py's planted duals): D reduced costs
    that differ only in their last bits sit at the top, far more than 8192 of them."""
    S, D, K = 700, 20000, 1024
    rng = np.random.default_rng(3)
    M = rng.random((S, D)) + 0.5
    a = rng.random(S)
    b = (M + a[:, None]).min(axis=0)
    y = np.concatenate([a, b + 0.01])
    rc_ref = orc.reduced_costs_ot(M, y)
    cnt, mn, ids, vals = orc.price_summary(rc_ref, K=K)
    assert cnt >= D
    pr = dev.Pricer(torch.device("cuda"), K)
    if fused_mode == "fused":
        res = price_in_one_fused_launch(dev, pr, M, y, K)
    else:
        res = dev.price_dense_ot(cu(M), cu(y), K=K, pricer=pr)
    assert pr.status == 0 and res.n_violating == cnt and res.min_rc == mn
    assert np.array_equal(res.topk_id, ids) and np.array_equal(res.topk_rc, vals)


@pytest.mark.parametrize("layout", ["ties", "tie_block"])
def test_fused_selection_refines_on_a_small_grid(dev, layout):
    """S = 16, D = 2560 is 10 tiles, so the fused kernel runs on 10 CTAs (2 560 selecting threads).  All
    40 960 reduced costs lie in one histogram bin and rank K falls inside a run of exact ties, next to
    near-ties that differ from them in low mantissa bits.  "ties": 600 near-ties below a tie of all the
    other arcs, refined down to the arc id; "tie_block": 900 near-ties below a tie of 3 000 arcs and the
    rest above it, which leaves 3 900 survivors -- more than the grid has threads -- for the rank.  The
    oracle's top K must come back from one launch, on both selection states of the pricer."""
    S, D, K = 16, 2560, 1024
    rng = np.random.default_rng(16)
    tie = -(1.0 + 2.0 ** -9)                                      # middle of its 0.4 %-wide histogram bin
    near = rng.integers(1 << 20, 1 << 30, S * D) * 2.0 ** -52
    side = np.zeros(S * D)                                        # -1: below the tie (more violating), +1: above
    pick = rng.permutation(S * D)
    if layout == "ties":
        side[pick[:600]] = -1
    else:
        side[pick[:900]] = -1
        side[pick[3900:]] = 1
    M = (3.0 + tie + side * near).reshape(S, D)
    y = np.concatenate([np.zeros(S), np.full(D, 3.0)])            # rc = M - 3
    rc_ref = orc.reduced_costs_ot(M, y)
    assert np.array_equal(rc_ref, tie + side * near)
    cnt, mn, ids, vals = orc.price_summary(rc_ref, K=K)
    assert cnt == S * D and vals[-1] == tie and vals[0] < tie     # rank K lies inside the tie
    pr = dev.Pricer(torch.device("cuda"), K, fused=True)
    for _ in range(2):
        res = price_in_one_fused_launch(dev, pr, M, y, K)
        assert pr.status == 0 and res.n_violating == cnt and res.min_rc == mn
        assert np.array_equal(res.topk_id, ids) and res.topk_rc.tobytes() == vals.tobytes()


def test_price_bins_are_monotone_over_magnitudes(dev, fused_mode):
    """Violations spread over 12 orders of magnitude, both signs of the exponent, with K landing
    inside a dense cluster: exercises the two-level histogram scan."""
    S, D = 512, 1024
    rng = np.random.default_rng(11)
    mag = 10.0 ** rng.uniform(-5.5, 6.5, size=(S, D))
    M = np.where(rng.random((S, D)) < 0.2, -mag, mag)
    M.ravel()[rng.choice(S * D, 3000, replace=False)] = -3.0e6        # a cluster of exact ties around rank 200..3200
    y = np.zeros(S + D)
    rc_ref = orc.reduced_costs_ot(M, y)
    for K in (1, 37, 1024):
        cnt, mn, ids, vals = orc.price_summary(rc_ref, K=K)
        res = dev.price_dense_ot(cu(M), cu(y), K=K)
        assert res.n_violating == cnt and res.min_rc == mn
        assert np.array_equal(res.topk_id, ids) and np.array_equal(res.topk_rc, vals)


def test_price_tma_stage_release_under_atomic_pressure(dev, fused_mode):
    """Every arc violates and all reduced costs fall into one histogram bin, so nothing is pruned and
    every warp-tile appends ~500 candidates (global atomics + stores saturate the load/store queue).
    The TMA pipeline must still hand out intact tiles: a stage may only be released once its data has
    ARRIVED in registers (regression: releasing after the shared loads were merely issued let the
    producer overwrite tiles still being read)."""
    S, D, K = 2000, 4096, 1024
    rng = np.random.default_rng(21)
    M = 1.0 + 1e-6 * rng.random((S, D))
    y = np.concatenate([np.zeros(S), np.full(D, 2.0)])              # rc in [-1, -1 + 1e-6]
    rc_ref = orc.reduced_costs_ot(M, y)
    cnt, mn, ids, vals = orc.price_summary(rc_ref, K=K)
    assert cnt == S * D
    pr = dev.Pricer(torch.device("cuda"), K, cand_cap=S * D)
    for _ in range(3):
        rc = torch.empty(S * D, dtype=torch.float64, device="cuda")
        pr.reset()
        pr.price_dense(cu(M), D, 0, S, D, cu(y[:S]), cu(y[S:]), rc_out=rc, variant=0)
        pr.select()
        res = pr.fetch()
        assert rc.cpu().numpy().tobytes() == rc_ref.tobytes()
        assert res.n_violating == cnt and res.min_rc == mn
        assert np.array_equal(res.topk_id, ids) and np.array_equal(res.topk_rc, vals)
        pr.reset()
        pr.price_dense(cu(M), D, 0, S, D, cu(y[:S]), cu(y[S:]), variant=0)      # same without the rc output
        pr.select()
        res = pr.fetch()
        assert res.n_violating == cnt and np.array_equal(res.topk_id, ids)
    if fused_mode == "fused":
        # the same pressure inside the fused kernel, whose selection refines the 8 M candidates of the one
        # bin in the same launch
        for _ in range(3):
            res = price_in_one_fused_launch(dev, pr, M, y, K)
            assert pr.status == 0 and res.n_violating == cnt and res.min_rc == mn
            assert np.array_equal(res.topk_id, ids) and np.array_equal(res.topk_rc, vals)


def test_price_row_slabs_and_merge(dev):
    """Row-sharded pricing: G slabs priced separately, per-slab top-K merged == single pass."""
    S, D, K, G = 1000, 768, 128, 4
    s, d, M = cases.ot_points(S, D, 77)
    y = cases.planted_duals(M, 77, 0.05)
    Mt, yt = cu(M), cu(y)
    whole = dev.price_dense_ot(Mt, yt, K=K)
    blocks_rc, blocks_id, total = [], [], 0
    rows = S // G
    for g in range(G):
        pr = dev.Pricer(torch.device("cuda"), K)
        pr.reset()
        pr.price_dense(Mt[g * rows:(g + 1) * rows], D, g * rows, rows, D, yt[g * rows:(g + 1) * rows], yt[S:])
        pr.select()
        r = pr.fetch()
        total += r.n_violating
        blocks_rc.append(pr.out_rc.clone())
        blocks_id.append(pr.out_id.clone())
    out_rc, out_id, out_n = dev.topk_merge(torch.stack(blocks_rc), torch.stack(blocks_id))
    k = int(out_n.item())
    assert total == whole.n_violating
    assert np.array_equal(out_id[:k].cpu().numpy(), whole.topk_id)
    assert np.array_equal(out_rc[:k].cpu().numpy(), whole.topk_rc)


def test_topk_merge_above_the_one_thread_per_element_size(dev):
    """sx_topk_merge with G * K > 2^22 (5 blocks of 2^20, 84 MB as an all-gathered (G, 2K + 4) buffer) runs the
    prefix bound + rank merge.  Sorted, padded blocks with many rc ties, tails of padding and one block that is
    all padding, against a NumPy lexsort of all real entries; the pricing headers fold into the summary."""
    G, K = 5, 1 << 20
    rng = np.random.default_rng(2024)
    for n_real in ([K, K - 12345, 0, K // 3, 777], [1000, 0, 0, 5000, 3]):
        ids_all = rng.permutation(sum(n_real)).astype(np.int64) * 3 + 7      # distinct across blocks
        buf = np.zeros((G, 2 * K + 4), dtype=np.int64)
        rc_real, id_real, off = [], [], 0
        for g, n in enumerate(n_real):
            rc = -1.0 - np.round(rng.random(n) * 1000) / 1000                # about a thousand distinct values
            ids = ids_all[off:off + n]
            off += n
            o = np.lexsort((ids, rc))
            buf[g, :K] = np.float64(np.inf).view(np.int64)
            buf[g, K:2 * K] = -1
            buf[g, :n] = rc[o].view(np.int64)
            buf[g, K:K + n] = ids[o]
            buf[g, 2 * K:] = [n, rng.integers(-1000, 1000), 0, 8 * (g == 1)]  # n_violating, min key, -, status
            rc_real.append(rc)
            id_real.append(ids)
        rc_real, id_real = np.concatenate(rc_real), np.concatenate(id_real)
        o = np.lexsort((id_real, rc_real))[:K]
        gathered = cu(buf)
        out_rc, out_id, out_n, summary = dev.topk_merge(gathered[:, :K].view(torch.float64), gathered[:, K:2 * K],
                                                        gathered[:, 2 * K:])
        k = int(out_n.item())
        assert k == o.size
        assert np.array_equal(out_id[:k].cpu().numpy(), id_real[o])
        assert out_rc[:k].cpu().numpy().tobytes() == rc_real[o].tobytes()
        assert np.all(out_id[k:].cpu().numpy() == -1) and np.all(np.isinf(out_rc[k:].cpu().numpy()))
        hdr = buf[:, 2 * K:]
        assert summary.cpu().numpy().tolist() == [int(hdr[:, 0].sum()), int(hdr[:, 1].min()), int(hdr[:, 0].max()), 8]


@pytest.mark.parametrize("G,K", [(2, 128), (8, 1024), (5, 33)])
def test_ll_exchange_and_merge_with_emulated_ranks(dev, G, K):
    """The flag-in-data exchange on one GPU: G buffers stand for G ranks, every "rank" pushes its block
    into all of them (a push never waits), then the merge polls / stages / ranks out of buffer 0.
    Result == sx_topk_merge on the same blocks == the oracle's global top-K.  Two epochs (both halves)."""
    import ctypes
    from smart_crossover._native import check, lib
    S, D = 64 * G, 700
    s, d, M = cases.ot_points(S, D, 5 + G)
    Mt = cu(M)
    blk = 2 * K + dev.Pricer.BLOCK_TAIL
    nbytes = lib.sx_exchange_ll_buffer_bytes(blk, G)
    bufs = [torch.zeros(nbytes // 8, dtype=torch.int64, device="cuda") for _ in range(G)]
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    rows = S // G
    for epoch, noise in ((1, 0.05), (2, 0.2)):
        y = cases.planted_duals(M, 7 * epoch, noise)
        yt = cu(y)
        whole = dev.price_dense_ot(Mt, yt, K=K)
        blocks = []
        for g in range(G):
            pr = dev.Pricer(torch.device("cuda"), K)
            pr.reset()
            pr.price_dense(Mt[g * rows:(g + 1) * rows], D, g * rows, rows, D, yt[g * rows:(g + 1) * rows], yt[S:])
            pr.select()
            blocks.append(pr.block.clone())
            # rank g's view of the peers: entry g is its own buffer, which holds the epoch counter it reads
            ptrs = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device="cuda")
            check(lib.sx_exchange_push_ll(dev._ptr(blocks[-1]), blk, dev._ptr(ptrs), g, G, dev._stream()), "push")
        torch.cuda.synchronize()
        out = torch.zeros(2 * K + 6, dtype=torch.int64, device="cuda")
        check(lib.sx_topk_merge_ll(dev._ptr(bufs[0]), blk, G, K, dev._ptr(out[:K]), dev._ptr(out[K:2 * K]),
                                   dev._ptr(out[2 * K:]), dev._ptr(out[2 * K + 1:]), dev._ptr(status), dev._stream()),
              "merge_ll")
        h = out.cpu().numpy()
        k = int(h[2 * K])
        assert int(status.item()) == 0 and k == whole.topk_id.size
        assert np.array_equal(h[K:K + k], whole.topk_id) and np.array_equal(h[:k].view(np.float64), whole.topk_rc)
        assert int(h[2 * K + 1]) == whole.n_violating and h[2 * K + 2] == np.float64(whole.min_rc).view(np.int64) \
            or lib.sx_key_to_f64(int(h[2 * K + 2])) == whole.min_rc
        assert int(h[2 * K + 4]) == 0 and np.all(h[K + k:2 * K] == -1)
        # the plain merge on the same blocks agrees
        stack = torch.stack(blocks)
        o_rc, o_id, o_n = dev.topk_merge(stack[:, :K].view(torch.float64), stack[:, K:2 * K])
        assert int(o_n.item()) == k and np.array_equal(o_id[:k].cpu().numpy(), whole.topk_id)


@pytest.mark.parametrize("G,K", [(2, 128), (8, 1024), (5, 33), (3, 1)])
def test_fused_pass_pushes_to_emulated_ranks(dev, G, K):
    """sx_price_dense_ot_fused with G emulated ranks on one GPU: every "rank" prices its row slab, selects and
    stores its block straight into all G exchange buffers from inside the pricing kernel; every rank's merge
    then finds all G blocks in its own buffer.  Five passes on the same pricers (both selection states, both
    buffer halves, a converged pass with only padding, a pass where most arcs violate)."""
    from smart_crossover._native import check, lib
    S, D = 64 * G + 3, 700
    s, d, M = cases.ot_points(S, D, 50 + G)
    Mt = cu(M)
    blk = 2 * K + dev.Pricer.BLOCK_TAIL
    nbytes = lib.sx_exchange_ll_buffer_bytes(blk, G)
    bufs = [torch.zeros(nbytes // 8, dtype=torch.int64, device="cuda") for _ in range(G)]
    ptrs = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device="cuda")
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    bounds = [S * g // G for g in range(G + 1)]
    pricers = [dev.Pricer(torch.device("cuda"), K, fused=True) for _ in range(G)]
    ys = [cases.planted_duals(M, 7, 0.05), cases.planted_duals(M, 8, 0.3),
          cases.planted_duals(M, 9, 0.0) - np.concatenate([np.zeros(S), np.full(D, 1e-3)]),
          np.concatenate([np.zeros(S), np.full(D, 1.0)]), cases.planted_duals(M, 10, 0.01)]
    for y in ys:
        yt = cu(y)
        cnt, mn, ids, vals = orc.price_summary(orc.reduced_costs_ot(M, y), K)
        for g in range(G):
            r0, r1 = bounds[g], bounds[g + 1]
            pricers[g].price_dense_fused(Mt[r0:r1], D, r0, r1 - r0, D, yt[r0:r1], yt[S:], peer_bufs=dev._ptr(ptrs),
                                         rank=g, G=G)
        for g in range(G):
            out = torch.zeros(2 * K + 6, dtype=torch.int64, device="cuda")
            check(lib.sx_topk_merge_ll(dev._ptr(bufs[g]), blk, G, K, dev._ptr(out[:K]), dev._ptr(out[K:2 * K]),
                                       dev._ptr(out[2 * K:]), dev._ptr(out[2 * K + 1:]), dev._ptr(status),
                                       dev._stream()), "merge_ll")
            h = out.cpu().numpy()
            k = int(h[2 * K])
            assert int(status.item()) == 0 and k == ids.size
            assert np.array_equal(h[K:K + k], ids) and h[:k].view(np.float64).tobytes() == vals.tobytes()
            assert int(h[2 * K + 1]) == cnt and lib.sx_key_to_f64(int(h[2 * K + 2])) == mn
            assert int(h[2 * K + 4]) == 0 and np.all(h[K + k:2 * K] == -1)
        # the local blocks hold each slab's own top-K
        for g in range(G):
            r0, r1 = bounds[g], bounds[g + 1]
            c_g, m_g, i_g, v_g = orc.price_summary(orc.reduced_costs_ot(M[r0:r1], np.concatenate([y[r0:r1], y[S:]])), K)
            res = pricers[g].fetch()
            assert res.n_violating == c_g and res.min_rc == m_g and pricers[g].status == 0
            assert np.array_equal(res.topk_id, i_g + r0 * D) and res.topk_rc.tobytes() == v_g.tobytes()


@pytest.mark.parametrize("K", [1, 64, 1024])
def test_fused_pass_in_kernel_merge_of_one_block(dev, K):
    """The in-kernel merge with G = 1 (the only form one GPU can run: with G > 1 every rank's kernel waits
    for the others' pushes; tests/test_gpu_multirank.py covers that on real ranks): the block pushed into
    the rank's own exchange buffer comes back merged, over several epochs."""
    from smart_crossover._native import lib
    S, D = 300, 1024
    s, d, M = cases.ot_points(S, D, 91)
    Mt = cu(M)
    blk = 2 * K + dev.Pricer.BLOCK_TAIL
    buf = torch.zeros(lib.sx_exchange_ll_buffer_bytes(blk, 1) // 8, dtype=torch.int64, device="cuda")
    ptrs = torch.tensor([buf.data_ptr()], dtype=torch.int64, device="cuda")
    merged = torch.zeros(2 * K + 6, dtype=torch.int64, device="cuda")
    xstatus = merged[2 * K + 5:].view(torch.int32)[:1]
    pr = dev.Pricer(torch.device("cuda"), K, fused=True)
    assert lib.sx_fused_merge_fits(K, 1)
    for it, noise in enumerate([0.05, 0.3, 0.0, 0.01, 0.3]):
        y = cases.planted_duals(M, 20 + it, noise)
        if noise == 0.0:
            y[S:] -= 1e-3
        yt = cu(y)
        cnt, mn, ids, vals = orc.price_summary(orc.reduced_costs_ot(M, y), K)
        pr.price_dense_fused(Mt, D, 0, S, D, yt[:S], yt[S:], peer_bufs=dev._ptr(ptrs), rank=0, G=1, merged=merged,
                             xstatus=xstatus)
        h = merged.cpu().numpy()
        k = int(h[2 * K])
        assert k == ids.size and int(h[2 * K + 5]) == 0 and int(h[2 * K + 4]) == 0
        assert np.array_equal(h[K:K + k], ids) and h[:k].view(np.float64).tobytes() == vals.tobytes()
        assert int(h[2 * K + 1]) == cnt and lib.sx_key_to_f64(int(h[2 * K + 2])) == mn and int(h[2 * K + 3]) == cnt
        assert np.all(h[K + k:2 * K] == -1)


@pytest.mark.parametrize("K", [0, 1, 100, 1024])
def test_fused_pass_sequence_on_one_pricer(dev, K):
    """Passes alternate between the pricer's two selection states; each pass clears the other one.  A long
    sequence of very different duals on ONE pricer must give the oracle's answer every time (a stale
    histogram bin or counter would prune real candidates)."""
    S, D = 1500, 2048
    rng = np.random.default_rng(K)
    M = rng.random((S, D))
    Mt = cu(M)
    pr = dev.Pricer(torch.device("cuda"), K, fused=True)
    assert pr.fused
    fracs = [0.5, 1e-4, 0.0, 0.9, 0.02, 0.0, 1e-5, 0.3, 0.3, 1.0]
    for it, frac in enumerate(fracs):
        y = np.concatenate([rng.normal(0, 1e-3, S), np.full(D, frac - 1e-4)])      # rc ~ M - frac
        res = dev.price_dense_ot(Mt, cu(y), K=K, pricer=pr)
        cnt, mn, ids, vals = orc.price_summary(orc.reduced_costs_ot(M, y), K)
        # dense violations put more than 4096 candidates into the K-th value's histogram bin: those passes are
        # repeated by the separate kernels (and the fused state must survive that); the others stay fused
        assert pr.status == 0 and (pr._last_fused or frac > 0.02), f"pass {it} fell back"
        assert res.n_violating == cnt and res.min_rc == mn, f"pass {it}"
        assert np.array_equal(res.topk_id, ids) and res.topk_rc.tobytes() == vals.tobytes(), f"pass {it}"


@pytest.mark.parametrize("E,off", [(100003, 0), (4096, 0), (7, 0), (50001, 1), (50002, 2)])
def test_price_arcs_vector_and_scalar_paths(dev, E, off):
    """Arc-list pricing takes 128-bit loads over the bulk of 16-byte aligned arrays and scalar loads for the last
    < 4 arcs or misaligned views (`off` shifts every array by that many elements): same reduced costs (bitwise),
    count, min and top-K either way."""
    N, K = 5000, 100
    rng = np.random.default_rng(E + off)
    tail = rng.integers(0, N, E + off).astype(np.int32)
    head = ((tail + 1 + rng.integers(0, N - 1, E + off)) % N).astype(np.int32)
    c = rng.integers(1, 100, E + off).astype(np.float64)
    y = rng.random(N) * 60.0
    vb = rng.choice(np.array([-1, -2, 0], dtype=np.int8), E + off, p=[0.8, 0.1, 0.1])
    ct, tt, ht, vt = cu(c)[off:], cu(tail)[off:], cu(head)[off:], cu(vb)[off:]
    rc_ref = orc.reduced_costs_arcs(c[off:], tail[off:], head[off:], y, vb[off:])
    cnt, mn, ids, vals = orc.price_summary(rc_ref, K)
    res = dev.price_arcs(ct, tt, ht, cu(y), vbasis=vt, K=K, want_rc=True)
    assert res.rc.cpu().numpy().tobytes() == rc_ref.tobytes()
    assert res.n_violating == cnt and res.min_rc == mn
    assert np.array_equal(res.topk_id, ids) and res.topk_rc.tobytes() == vals.tobytes()
    res = dev.price_arcs(ct, tt, ht, cu(y), vbasis=None, K=K)              # no basis statuses
    cnt, mn, ids, vals = orc.price_summary(orc.reduced_costs_arcs(c[off:], tail[off:], head[off:], y), K)
    assert res.n_violating == cnt and np.array_equal(res.topk_id, ids)


@pytest.mark.parametrize("name", MCF_FULL)
def test_mcf_scores_queue_and_arc_pricing_golden(dev, name):
    import scipy.sparse as sp
    fx = Fixture(name)
    tail, head, b, c, u, x = (fx.inp[k] for k in ("tail", "head", "b", "c", "u", "x"))
    N, E = b.size, c.size
    A = sp.csr_matrix((np.concatenate([np.ones(E), -np.ones(E)]),
                       (np.concatenate([tail, head]), np.concatenate([np.arange(E)] * 2))), shape=(N, E))
    A.sort_indices()
    ind = dev.score_mcf(cu(x), cu(u), cu(tail, torch.int32), cu(head, torch.int32), cu(A.indptr, torch.int64),
                        cu(A.indices, torch.int32), cu(A.data, torch.int8))
    assert ind.cpu().numpy().tobytes() == fx.out["scores"].tobytes()
    order, skey, queue, korder = sort_pipeline(dev, ind)
    assert np.array_equal(queue.cpu().numpy(), fx.out["queue"])
    res = dev.price_arcs(cu(c), cu(tail, torch.int32), cu(head, torch.int32), cu(fx.out["y"]),
                         vbasis=cu(fx.out["vbasis"], torch.int8), K=32, want_rc=True)
    assert res.rc.cpu().numpy().tobytes() == fx.out["rc"].tobytes()
    cnt, mn, ids, vals = orc.price_summary(fx.out["rc"], K=32)
    assert res.n_violating == cnt and res.min_rc == mn and res.optimal == bool(fx.out["optimal"])
    assert np.array_equal(res.topk_id, ids) and np.array_equal(res.topk_rc, vals)


def test_mcf_mid_digests(dev):
    import scipy.sparse as sp
    tail, head, b, c, u, x = mcf_mid_inputs()
    dg = digests()["mcf_mid_20k"]["digests"]
    N, E = b.size, c.size
    A = sp.csr_matrix((np.concatenate([np.ones(E), -np.ones(E)]),
                       (np.concatenate([tail, head]), np.concatenate([np.arange(E)] * 2))), shape=(N, E))
    A.sort_indices()
    ind = dev.score_mcf(cu(x), cu(u), cu(tail, torch.int32), cu(head, torch.int32), cu(A.indptr, torch.int64),
                        cu(A.indices, torch.int32), cu(A.data, torch.int8))
    assert cases.digest(ind.cpu().numpy()) == dg["scores"]
    order, skey, queue, korder = sort_pipeline(dev, ind)
    assert cases.digest(queue.cpu().numpy()) == dg["queue"]
    small = Fixture("mcf_mid_20k_small").out
    vb = np.zeros(E, dtype=np.int8)   # digest of rc was taken with the stored vbasis; count only here
    res = dev.price_arcs(cu(c), cu(tail, torch.int32), cu(head, torch.int32), cu(small["y"]), K=0)
    rc = orc.reduced_costs_arcs(c, tail, head, small["y"])
    assert res.n_violating == int((rc < -1e-6).sum())


# ---- full-size property tests (BASELINE.json configs[3]: 20 000 x 20 000, 3.2 GB) -------------------
def test_c4_full_size_planted_violators(dev, fused_mode):
    """No oracle pass at this size: plant a known set of violators into a dual-feasible instance
    and require the pricing pass to return exactly that set, in order."""
    S = D = 20000
    g = torch.Generator(device="cuda").manual_seed(20260004)
    P = torch.rand(S, 2, generator=g, device="cuda", dtype=torch.float64)
    Q = torch.rand(D, 2, generator=g, device="cuda", dtype=torch.float64)
    M = torch.empty(S, D, dtype=torch.float64, device="cuda")
    for r0 in range(0, S, 2000):
        dx = P[r0:r0 + 2000, 0:1] - Q[None, :, 0]
        dy = P[r0:r0 + 2000, 1:2] - Q[None, :, 1]
        M[r0:r0 + 2000] = dx * dx + dy * dy
    a = torch.rand(S, generator=g, device="cuda", dtype=torch.float64)
    b = torch.full((D,), float("inf"), dtype=torch.float64, device="cuda")
    for r0 in range(0, S, 2000):
        b = torch.minimum(b, (M[r0:r0 + 2000] + a[r0:r0 + 2000, None]).min(dim=0).values)
    b = b - 1e-3                                  # strictly feasible: rc >= 1e-3 everywhere
    y = torch.cat([a, b])
    res = dev.price_dense_ot(M, y, K=512)
    assert res.optimal and res.n_violating == 0 and res.min_rc >= 1e-3 - 1e-12
    # plant 300 violators with distinct, known reduced costs
    rng = np.random.default_rng(4)
    ids = np.sort(rng.choice(S * D, size=300, replace=False))
    i, j = ids // D, ids % D
    want_rc = -(1.0 + rng.permutation(300).astype(np.float64))      # -1 .. -300
    yi, yj = a[cu(i)], b[cu(j)]
    M[cu(i), cu(j)] = cu(want_rc) + (yj - yi)
    got = dev.price_dense_ot(M, y, K=512)
    rc_exact = (M[cu(i), cu(j)] - (yj - yi)).cpu().numpy()
    o = np.lexsort((ids, rc_exact))
    assert got.n_violating == 300
    assert np.array_equal(got.topk_id, ids[o]) and np.array_equal(got.topk_rc, rc_exact[o])
    assert got.min_rc == rc_exact.min()
    for variant in (1, 2):
        alt = dev.price_dense_ot(M, y, K=512, variant=variant)
        assert alt.n_violating == 300 and np.array_equal(alt.topk_id, got.topk_id)


def test_c5_full_size_arc_ids_beyond_2_31(dev):
    """BASELINE.json configs[4]: 60 000 x 60 000 (28.8 GB, 3.6e9 arcs: ids past 2^31, where int32 indexing breaks).  A constant cost
    matrix with zero duals prices to rc = 1 everywhere; 3 000 planted negative entries (most of them in
    the last rows, where arc ids exceed 2^31) must come back exactly, in order, through the TMA path,
    and row slabs priced separately must merge to the same answer."""
    free, _ = torch.cuda.mem_get_info()
    S = D = 60000
    if free < 8 * S * D + (4 << 30):
        pytest.skip("needs ~33 GB of free device memory")
    M = torch.ones(S, D, dtype=torch.float64, device="cuda")
    y = torch.zeros(S + D, dtype=torch.float64, device="cuda")
    rng = np.random.default_rng(60)
    rows = np.concatenate([rng.integers(0, S, 500), rng.integers(S - 4000, S, 2500)])
    cols = rng.integers(0, D, rows.size)
    ids = np.unique(rows.astype(np.int64) * D + cols)
    vals = -(1.0 + rng.permutation(ids.size)).astype(np.float64) / 7.0          # distinct, not dyadic
    M.view(-1)[cu(ids)] = cu(vals)
    K = 1024
    res = dev.price_dense_ot(M, y, K=K)
    o = np.argsort(vals, kind="stable")[:K]
    assert ids.max() > (1 << 31) and res.n_violating == ids.size and res.min_rc == vals.min()
    assert np.array_equal(res.topk_id, ids[o]) and np.array_equal(res.topk_rc, vals[o])
    # two row slabs (as two ranks would hold them), merged
    blocks_rc, blocks_id = [], []
    for r0, r1 in ((0, 31000), (31000, S)):
        pr = dev.Pricer(torch.device("cuda"), K)
        pr.reset()
        pr.price_dense(M[r0:r1], D, r0, r1 - r0, D, y[r0:r1], y[S:])
        pr.select()
        torch.cuda.synchronize()
        blocks_rc.append(pr.out_rc.clone())
        blocks_id.append(pr.out_id.clone())
    m_rc, m_id, m_n = dev.topk_merge(torch.stack(blocks_rc), torch.stack(blocks_id))
    assert int(m_n.item()) == K and np.array_equal(m_id.cpu().numpy(), ids[o])
    del M


def test_kruskal_prefix_large_properties(dev):
    """1.3e8 weights: the head returned by sx_kruskal_prefix is sorted (descending weight, ties by
    ascending id), holds at least T arcs, and nothing outside it is heavier than its lightest arc."""
    n, T = 1 << 27, 500000
    g = torch.Generator(device="cuda").manual_seed(11)
    w = torch.rand(n, generator=g, device="cuda", dtype=torch.float64) ** 8       # skewed toward 0, like scores
    w[::1000003] = 0.75                                                           # a run of exact ties near the top
    head = dev.kruskal_prefix(w, T)
    assert head is not None
    idx = head.to(torch.int64) & 0xFFFFFFFF
    hw = w[idx]
    assert idx.numel() >= T and idx.unique().numel() == idx.numel()
    assert bool((hw[1:] <= hw[:-1]).all())
    same = hw[1:] == hw[:-1]
    assert bool((idx[1:][same] > idx[:-1][same]).all())
    rest = torch.ones(n, dtype=torch.bool, device="cuda")
    rest[idx] = False
    assert float(w[rest].max()) < float(hw[-1])


@pytest.mark.parametrize("threads,n", [(2, 1 << 25), (1024, (1 << 25) + 12345), (512, 3_000_001), (1024, 3_000_001),
                                       (256, 1_300_000), (384, 1_300_000)])
def test_large_sort_properties(dev, threads, n):
    """Output is a permutation, keys non-decreasing, ties in ascending id -- for every downsweep tile shape
    (`threads`; 2 = chosen by size; 1024 is what inputs of 2^26 keys and more take), partial last tiles included."""
    from smart_crossover._native import lib
    assert lib.sx_sort_set_tuning(threads) == 0 and lib.sx_sort_set_tuning(0) == 0     # launches per pass
    try:
        _large_sort_properties(dev, n)
    finally:
        assert lib.sx_sort_set_tuning(2) == 0 and lib.sx_sort_set_tuning(1) == 0


def _large_sort_properties(dev, n):
    g = torch.Generator(device="cuda").manual_seed(7)
    key = torch.randint(0, 1 << 20, (n,), generator=g, device="cuda").to(torch.float64) / 1024.0
    order, skey = dev.argsort_f64(key)
    idx = order.to(torch.int64) & 0xFFFFFFFF
    assert torch.equal(key[idx], skey)
    assert bool((skey[1:] >= skey[:-1]).all())
    same = skey[1:] == skey[:-1]
    assert bool((idx[1:][same] > idx[:-1][same]).all())
    assert int(torch.bincount(idx, minlength=n).max().item()) == 1


# ---- full-size MCF (BASELINE.json configs[2]: NETGEN-style 1M nodes / 10M arcs) ------------------------
def test_c3_full_size_mcf_path(dev):
    """Scores, queue, spanning forest, potentials and arc pricing on the 1M-node / 10M-arc instance,
    against the oracle (bit-exact scores / order / forest / reduced costs; potentials 1e-9)."""
    import scipy.sparse as sp
    N, E = 1_000_000, 10_000_000
    tail, head, b, c, u = cases.netgen_like(N, E, 20260003)
    x = cases.mcf_interior_flow(u, 20260003)
    A = sp.csr_matrix((np.concatenate([np.ones(E, np.int8), -np.ones(E, np.int8)]),
                       (np.concatenate([tail, head]), np.concatenate([np.arange(E)] * 2))), shape=(N, E))
    A.sort_indices()
    t32, h32 = cu(tail, torch.int32), cu(head, torch.int32)
    ind = dev.score_mcf(cu(x), cu(u), t32, h32, cu(A.indptr, torch.int64), cu(A.indices, torch.int32),
                        cu(A.data, torch.int8))
    ind_ref = orc.mcf_flow_scores(x, u, A)
    assert ind.cpu().numpy().tobytes() == ind_ref.tobytes()
    order, skey, queue, korder = sort_pipeline(dev, ind)
    assert np.array_equal(queue.cpu().numpy(), orc.stable_queue(ind_ref))
    ko_ref = orc.kruskal_order(ind_ref)
    assert np.array_equal(u32(korder), ko_ref)
    tree, n_tree = dev.kruskal(korder, N, tail=t32, head=h32)
    nt = int(n_tree.item())
    forest_ref = orc.spanning_forest(ko_ref, N, tail=tail, head=head)
    assert nt == forest_ref.size == N - 1                 # the ring makes the graph connected
    assert np.array_equal(tree[:nt].cpu().numpy(), forest_ref)
    y = dev.tree_potentials(tree, nt, N, cu(c), N - 1, tail=t32, head=h32, plus=1)
    y_ref = orc.tree_potentials(tail[forest_ref], head[forest_ref], c[forest_ref], N, N - 1)
    np.testing.assert_allclose(y.cpu().numpy(), y_ref, rtol=RTOL, atol=RTOL * np.abs(y_ref).max())
    vb = np.where(x > u / 2, -2, -1).astype(np.int8)
    res = dev.price_arcs(cu(c), t32, h32, cu(y_ref), vbasis=cu(vb), K=1000, want_rc=True)
    rc_ref = orc.reduced_costs_arcs(c, tail, head, y_ref, vb)
    assert res.rc.cpu().numpy().tobytes() == rc_ref.tobytes()
    cnt, mn, ids, vals = orc.price_summary(rc_ref, K=1000)
    assert res.n_violating == cnt and res.min_rc == mn
    assert np.array_equal(res.topk_id, ids) and np.array_equal(res.topk_rc, vals)


# ---- warm start ---------------------------------------------------------------------------------
@pytest.mark.parametrize("S,D,reg,iters", [(40, 40, 0.05, 200), (257, 130, 0.02, 500), (300, 1000, 10.0, 1000)])
def test_sinkhorn_warm_start_matches_sinkhorn_knopp(dev, S, D, reg, iters):
    """Device log-domain Sinkhorn == the Sinkhorn-Knopp iteration POT runs (oracle restatement), to
    1e-9 relative on the plan; marginals are met; the plan is a valid interior point for TNET."""
    from smart_crossover.warm_start import sinkhorn
    s, d, M = cases.ot_points(S, D, 40 + S)
    if reg >= 1.0:
        M = np.round(50 * M)                                       # MNIST-like integer costs with reg = 10
    X_ref, it_ref, err_ref = orc.sinkhorn_knopp(s, d, M, reg, iters, stop_thr=0.0)
    X, info = sinkhorn(s, d, M, reg, numItermax=iters, stopThr=0.0, log=True)
    assert info["niter"] == iters and X.shape == (S, D)
    np.testing.assert_allclose(X, X_ref, rtol=1e-9, atol=1e-300)
    np.testing.assert_allclose(X.sum(axis=1), s, rtol=1e-9)            # the last half-step fixes the rows
    assert np.all(X > 0)
    # with the stopping rule: stops early, within one check interval of the oracle, error below the threshold
    X2, info2 = sinkhorn(s, d, M, reg, numItermax=10000, stopThr=1e-7, log=True)
    _, it2, _ = orc.sinkhorn_knopp(s, d, M, reg, 10000, stop_thr=1e-7)
    assert info2["err"] < 1e-7 and abs(info2["niter"] - it2) <= 1

"""The fused pass over the lower-bound copy of the cost matrix (sx_cost_lb_build + sx_price_dense_ot_fused_lb):
the copy holds the high 32 bits of each fp64 cost rounded toward -inf, and a pass that streams it must return what the fp64 walk and the
oracle return, bit for bit -- count, minimum, status, top-K ids and reduced-cost bits.  Run on a B200:
`pytest -m gpu`."""
import numpy as np
import pytest

import cases
from oracle import network_oracle as orc

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
TOL = 1e-6
LB_MAX_FRAC = 1.0 / 2048        # kLbMaxViolatingFrac of sx_fused.cu: the walk after a pass above it is fp64


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from smart_crossover import device
    return device


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def lb_reference(M):
    """The copy's words from NumPy: the high half of each fp64 bit pattern, one unit away from zero for a
    negative value with a nonzero low half, quiet bit set for a NaN (uint32)."""
    b = np.ascontiguousarray(M, dtype=np.float64).view(np.uint64)
    hi, lo = (b >> np.uint64(32)).astype(np.uint32), (b & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    neg = (hi >> np.uint32(31)) == 1
    out = np.where((lo != 0) & neg, hi + np.uint32(1), hi)
    return np.where(np.isnan(M), hi | np.uint32(0x00080000), out).astype(np.uint32)


def lb_value(words):
    """The copy's words read back as the doubles the kernel compares with."""
    return (np.asarray(words, dtype=np.uint32).astype(np.uint64) << np.uint64(32)).view(np.float64)


def even_ld(M):
    """Device copy of M with an even leading dimension (the fused pass needs it): an (S, D) view."""
    S, D = M.shape
    t = torch.zeros(S, D + (D & 1), dtype=torch.float64, device="cuda")
    t[:, :D] = cu(M)
    return t[:, :D]


class Walks:
    """One fused pricer that streams the lower-bound copy and one that streams M, over the same matrix."""

    def __init__(self, dev, M, K, cand_cap=None):
        self.dev, self.M = dev, M
        self.S, self.D = M.shape
        self.Mt = even_ld(M)
        self.lb = dev.cost_lb(self.Mt)
        self.K = K
        self.p_lb = dev.Pricer(torch.device("cuda"), K, cand_cap=cand_cap, fused=True)
        self.p_64 = dev.Pricer(torch.device("cuda"), K, cand_cap=cand_cap, fused=True)

    def _pass(self, pr, yt, lb):
        S, D = self.S, self.D
        while True:
            pr.price_dense_fused(self.Mt, self.Mt.stride(0), 0, S, D, yt[:S], yt[S:S + D], TOL, lb=lb)
            res = pr.fetch()
            if not pr.overflowed(res):
                return res, pr.h_block.numpy().copy()
            pr.grow(res.n_violating)

    def price(self, y, expect_walk=None):
        yt = cu(y)
        r_lb, b_lb = self._pass(self.p_lb, yt, self.lb)
        walk = self.p_lb.fused_walk()
        r_64, b_64 = self._pass(self.p_64, yt, None)
        assert self.p_64.fused_walk() == 0
        if expect_walk is not None:
            assert walk == expect_walk
        # the whole block: K rc bits, K ids, count, min key, n_priced, status, n_out
        assert b_lb.tobytes() == b_64.tobytes()
        return r_lb, walk


def check_oracle(res, M, y, K):
    cnt, mn, ids, vals = orc.price_summary(orc.reduced_costs_ot(M, y), K)
    assert res.n_violating == cnt and res.min_rc == mn and res.status == 0
    assert np.array_equal(res.topk_id, ids) and res.topk_rc.tobytes() == vals.tobytes()


def test_cost_lb_build_matches_numpy(dev):
    """Special values, |x| > FLT_MAX, subnormals, odd D and row / column padding."""
    from smart_crossover._native import lib
    rng = np.random.default_rng(3)
    nan_low_payload = np.array([0x7FF0000000000001, 0xFFF0000000000001], dtype=np.uint64).view(np.float64)
    specials = np.array([*nan_low_payload, np.nan, np.inf, -np.inf, 0.0, -0.0, 1e-300, -1e-300, 1e-40, -1e-40, 3e-45, -3e-45,
                         5e-324, -5e-324, 1.7976931348623157e308, -1.7976931348623157e308, -0.5, 0.5, 1 + 2 ** -30,
                         -(1 + 2 ** -30),
                         1.5e-45, -1.5e-45, 4e38, -4e38, 3.4028234663852886e38, -3.4028234663852886e38,
                         3.4028235e38 * (1 + 1e-12), -3.4028235e38 * (1 + 1e-12), 1e308, -1e308,
                         0.1, -0.1, 1 / 3, -1 / 3, 1.0, -1.0, 16777217.0, -16777217.0])
    for S, D in [(7, 29), (33, 257), (5, 1), (130, 515)]:
        M = rng.normal(0, 1, (S, D)) * 10.0 ** rng.integers(-45, 39, (S, D))
        flat = M.ravel()
        flat[rng.choice(flat.size, min(flat.size, specials.size), replace=False)] = specials[:min(flat.size, specials.size)]
        Mt = even_ld(M)
        lb = dev.cost_lb(Mt)
        assert lb.stride(0) % 4 == 0 and lb.stride(0) >= D
        got = lb[:, :D].cpu().numpy().view(np.uint32)
        ref = lb_reference(M)
        assert got.tobytes() == ref.tobytes()
        L = lb_value(got)
        finite = ~np.isnan(M)
        assert np.all(L[finite] <= M[finite]) and np.all(np.isnan(L[~finite]))
    assert lib.sx_cost_lb_bytes(3, 5) == 3 * 8 * 4
    assert lib.sx_cost_lb_build(None, 4, 1, 4, None, 4, None) == -1


def _near_threshold(S, D, seed):
    """M with w = v - u = 0 everywhere (u = v = 0.25): rc = M.  Planted: arcs at exactly -tol and just above it
    whose copy rounds below -tol (flagged, not violators), arcs just below -tol (violators whose copy is the
    same value as a false positive's), and far violators."""
    rng = np.random.default_rng(seed)
    M = rng.random((S, D)) + 0.5
    w_below = lb_reference(np.array([-TOL]))[0]                        # largest copy value below -tol
    f_below, f_above = lb_value(w_below), lb_value(w_below - np.uint32(1))   # and the next one up
    assert f_below < -TOL < f_above
    flat = M.ravel()
    idx = rng.choice(flat.size, 400, replace=False)
    above = np.linspace(-TOL, f_above, 102)[1:-1]                     # rc > -tol, copy == f_below < -tol
    below = np.linspace(f_below, -TOL, 102)[1:-1]                     # rc < -tol, copy == f_below
    flat[idx[:100]] = above
    flat[idx[100:200]] = below
    flat[idx[200:220]] = -TOL
    flat[idx[220:]] = -rng.random(180)
    y = np.full(S + D, 0.25)
    assert np.all(lb_value(lb_reference(M[np.unravel_index(idx[:200], M.shape)])) == f_below)
    return M, y


@pytest.mark.parametrize("K", [1, 1024])
def test_false_positives_of_the_copy_are_not_counted(dev, K):
    M, y = _near_threshold(300, 1000, 11)
    w = Walks(dev, M, K)
    res, walk = w.price(y, expect_walk=1)
    check_oracle(res, M, y, K)
    assert res.n_violating == 100 + 180


@pytest.mark.parametrize("S,D", [(16, 256), (17, 257), (15, 255), (1, 1), (33, 513), (48, 768), (300, 1021)])
@pytest.mark.parametrize("K", [1, 1024])
def test_tile_boundary_shapes(dev, S, D, K):
    s, d, M = cases.ot_points(S, D, S * 1000 + D)
    y = cases.planted_duals(M, S + D, 0.02)
    w = Walks(dev, M, K)
    res, walk = w.price(y, expect_walk=1)
    check_oracle(res, M, y, K)


@pytest.mark.parametrize("K", [1, 1024])
def test_ties_at_the_kth_value(dev, K):
    """3 000 arcs share the K-th value exactly, next to near-ties one ulp away."""
    rng = np.random.default_rng(5)
    S, D = 400, 900
    M = rng.random((S, D)) + 0.5
    flat = M.ravel()
    b = K // 2                                      # arcs ahead of the ties: rank K falls among them
    idx = rng.choice(flat.size, b + 3200, replace=False)
    flat[idx[:b]] = -0.75
    flat[idx[b:b + 3000]] = -0.5
    flat[idx[b + 3000:b + 3100]] = np.nextafter(-0.5, 0.0)
    flat[idx[b + 3100:b + 3200]] = np.nextafter(-0.5, -1.0)
    y = np.full(S + D, 0.125)
    w = Walks(dev, M, K)
    res, _ = w.price(y, expect_walk=1)
    check_oracle(res, M, y, K)


@pytest.mark.parametrize("where", ["M_nan", "y_nan", "M_inf", "M_minf", "y_inf", "y_minf", "inf_minus_inf"])
def test_non_finite_costs_and_duals(dev, where):
    s, d, M = cases.ot_points(200, 600, 17)
    y = cases.planted_duals(M, 17, 0.01)
    S, D = M.shape
    if where == "M_nan":
        M[5, 7] = np.nan
    elif where == "y_nan":
        y[S + 9] = np.nan
    elif where == "M_inf":
        M[3, 100:110] = np.inf
    elif where == "M_minf":
        M[4, 200:203] = -np.inf
    elif where == "y_inf":
        y[11] = np.inf                      # w = v - inf = -inf: the whole row prices to +inf
    elif where == "y_minf":
        y[S + 13] = -np.inf                 # w = -inf - u: the column prices to +inf
    else:
        M[6, 50] = np.inf
        y[S + 50] = np.inf                  # inf - (inf - u) = NaN
    for K in (1, 64):
        w = Walks(dev, M, K)
        res, _ = w.price(y, expect_walk=1)
        rc = orc.reduced_costs_ot(M, y)
        cnt, _, ids, vals = orc.price_summary(rc, K)
        assert res.n_violating == cnt and np.array_equal(res.topk_id, ids) and res.topk_rc.tobytes() == vals.tobytes()
        assert res.has_nan == bool(np.isnan(rc).any())


def test_pass_without_violators(dev):
    """Only the minimum path: no arc violates, the minimum is an exact fp64 value the copy only bounds."""
    s, d, M = cases.ot_points(500, 1500, 23)
    y = cases.planted_duals(M, 23, 0.0)
    y[M.shape[0]:] -= 1e-3
    for K in (1, 1024):
        w = Walks(dev, M, K)
        res, _ = w.price(y, expect_walk=1)
        check_oracle(res, M, y, K)
        assert res.n_violating == 0 and res.min_rc > 0


def test_candidate_overflow_then_repeat(dev):
    """More violators than candidate slots: the pass overflows, the buffer grows and the pass is repeated (after a
    pass of more than 1/64 violators, the repeat streams M itself); both walks agree throughout."""
    s, d, M = cases.ot_points(600, 2000, 29)
    y = cases.planted_duals(M, 29, 0.3)
    w = Walks(dev, M, 1024, cand_cap=1024)
    res, walk = w.price(y)
    check_oracle(res, M, y, 1024)
    assert w.p_lb.cap > 1024 and walk == int(res.n_violating <= LB_MAX_FRAC * M.size)


def test_walk_choice_over_sparse_dense_sparse_passes(dev):
    """The walk of a pass follows the violator count of the previous pass on the same state: the first pass
    streams the copy, a pass after a dense one streams M, a pass after a sparse one the copy again."""
    rng = np.random.default_rng(31)
    S, D = 1500, 2048
    M = rng.random((S, D))
    w = Walks(dev, M, 100)
    fracs = [1e-4, 0.5, 0.5, 1e-4, 0.0, 1e-3, 0.3, 1e-5]
    prev = 0
    for it, frac in enumerate(fracs):
        y = np.concatenate([rng.normal(0, 1e-3, S), np.full(D, frac - 1e-4)])      # rc ~ M - frac
        res, walk = w.price(y, expect_walk=int(prev <= LB_MAX_FRAC * M.size))
        check_oracle(res, M, y, 100)
        prev = res.n_violating


@pytest.mark.parametrize("G,K", [(2, 128), (5, 33), (3, 1)])
def test_emulated_ranks_with_the_copy(dev, G, K):
    """G emulated ranks on one GPU, each pricing its slab through its own copy and pushing its block into every
    rank's exchange buffer: every rank's merge equals the oracle over the whole matrix."""
    from smart_crossover._native import check, lib
    S, D = 64 * G + 3, 700
    s, d, M = cases.ot_points(S, D, 70 + G)
    Mt = cu(M)
    blk = 2 * K + dev.Pricer.BLOCK_TAIL
    nbytes = lib.sx_exchange_ll_buffer_bytes(blk, G)
    bufs = [torch.zeros(nbytes // 8, dtype=torch.int64, device="cuda") for _ in range(G)]
    ptrs = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device="cuda")
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    bounds = [S * g // G for g in range(G + 1)]
    lbs = [dev.cost_lb(Mt[bounds[g]:bounds[g + 1]]) for g in range(G)]
    pricers = [dev.Pricer(torch.device("cuda"), K, fused=True) for _ in range(G)]
    ys = [cases.planted_duals(M, 7, 0.05), cases.planted_duals(M, 8, 0.3), cases.planted_duals(M, 10, 0.01)]
    for y in ys:
        yt = cu(y)
        cnt, mn, ids, vals = orc.price_summary(orc.reduced_costs_ot(M, y), K)
        for g in range(G):
            r0, r1 = bounds[g], bounds[g + 1]
            pricers[g].price_dense_fused(Mt[r0:r1], D, r0, r1 - r0, D, yt[r0:r1], yt[S:], peer_bufs=dev._ptr(ptrs),
                                         rank=g, G=G, lb=lbs[g])
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


def test_sharded_and_ot_pricers_hold_a_copy(dev):
    """ShardedDensePricer builds the copy and its passes stream it; OTPricer (sx_ot_pricer) returns the oracle's
    answer over several passes with its own copy."""
    from smart_crossover.network_methods.sharded import ShardedDensePricer
    s, d, M = cases.ot_points(700, 1200, 37)
    S, D = M.shape
    sp = ShardedDensePricer(cu(M), S, 0, 64, TOL)
    assert sp.fused and sp.lb is not None and sp.lb.dtype == torch.int32
    hp = dev.OTPricer(dev.CostSlabs.from_host(M, [torch.cuda.current_device()]), 64)
    dense = np.concatenate([np.zeros(S), np.ones(D)])         # rc = M - 1: most arcs violate
    for y in [cases.planted_duals(M, 1, 0.01), dense, cases.planted_duals(M, 4, 0.001)]:
        for res in (sp.price(y), hp.price(y[:S], y[S:])):
            check_oracle(res, M, y, 64)
    assert sp.pricer.fused_walk() == 0           # after a dense pass
    hp.close()

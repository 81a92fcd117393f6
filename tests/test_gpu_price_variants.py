"""The dense OT pricing pass (sx_price_dense_ot) at every launch variant against a literal NumPy reference.

`bench.py` times variant 0, the TMA pipeline, at the default shape only; `bench.py --sweep` times every shape of
the table in sx_price.cu but checks no result.  Every shape and every variant computes
rc_ij = fl(M_ij - fl(y_dst[j] - y_src[i])) bit for bit, so the few lines of NumPy in `Ref` are an exact oracle for
all of them.  Reduced costs, the top-K reduced costs and the minimum are compared as bytes (NaN reduced costs by
position: IEEE fixes no NaN payload); ids, counts and the status word exactly.  No tolerance is used anywhere.

  * Variant 0 at each of the 14 TMA shapes (rows per box, ring stages, consumer warps, CTAs per SM), with and
    without rc_out: a boundary grid of S_loc around the shape's box height and D around the 256-column box width,
    and a 6000 x 4099 matrix on which every CTA wraps its stage ring at least four times, at K = 1 and K = 1024 and
    through the candidate-overflow repeat.  The cache hints of the TMA loads (L2 promotion, evict-first) at shape 6
    and at a 16-warp shape.
  * Variants 1 and 2, the direct-load kernels, at 1 - 40 CTAs per SM, with D chosen so that the grid is smaller
    than, equal to, a multiple of, and neither of the number of column blocks; variant 2 on an 8-byte offset base.
  * The score kernel compiled for 3 CTAs per SM (sx_score_set_tuning(3)), scores and the 4096-bin key histogram.

Every matrix is a row slab of a padded buffer (ld > D, NaN padding and NaN rows around it, row0 > 0 with arc ids
straddling 2^31), and rc_out is written with ld_out > D into a buffer whose padding must stay untouched.  Planted in
every matrix: a run of exact ties at the K-th value that covers every row group of a tile and several tiles, so that
K cuts it and ids decide; rc = -tol exactly and its two neighbours; and in the special flavour NaN and +-inf costs
and duals, one NaN in the last row and last column of a tile.

The tuning setters are process-wide.  The `knobs` fixture restores the defaults -- shape 6, 16 direct CTAs per SM,
L2 promotion 3 with evict-first, 4 score CTAs per SM -- whatever a test does.  The tests without the `gpu` marker
check the reference against the golden fixtures, the case generator against what it claims to plant, and that the
setters reject out-of-range values.
"""
import ctypes
import functools

import numpy as np
import pytest

import cases
from golden_util import OT_FULL, Fixture, c2_inputs, digests
from oracle import network_oracle as orc

TOL = 1e-6                    # TOLERANCE_FOR_REDUCED_COSTS
INF, NAN = np.inf, np.nan
NAN_RC = 8                    # SX_STATUS_NAN_RC
ERR_INVALID, ERR_UNALIGNED = -1, -6
SENTINEL = -7.25              # fills rc_out padding; it must survive every pass

# sx_price.cu kTmaShapes: (rows per box, stages, consumer warps, CTAs per SM); the index is the shape's address
TMA_SHAPES = [
    (16, 6, 8, 1), (16, 6, 16, 1), (32, 3, 8, 1), (32, 3, 16, 1), (16, 7, 16, 1), (8, 12, 16, 1),
    (16, 3, 8, 2), (8, 6, 8, 2), (24, 4, 16, 1), (20, 5, 16, 1), (12, 9, 16, 1),
    (12, 4, 8, 2), (8, 7, 8, 2), (8, 4, 8, 3),
]
DEFAULT_SHAPE, DEFAULT_DIRECT_CTAS, DEFAULT_L2, DEFAULT_EVICT, DEFAULT_SCORE_CTAS = 6, 16, 3, 1, 4
BOX_COLS = 256                # TMA box width and column block of every variant
DIRECT_ROWS = 8               # rows per tile of the direct-load kernels
GRID_D = [1, 2, 255, 256, 257, 512, 1001]
LONG_S, LONG_D, LONG_LD = 6000, 4099, 4100
TIE_ROWS_LONG = 120           # tie rows of the long matrix: whole tiles of every box height but 32 (3.75 tiles)
ROW_ALL_TILES = 479           # last row of a tile for every box height (480 = lcm of 8, 12, 16, 20, 24, 32)


# ==== reference ============================================================================================
def rc_ref(M, y_src, y_dst):
    """rc_ij = fl(M_ij - fl(y_dst[j] - y_src[i])) in float64 (NumPy contracts nothing into an FMA)."""
    with np.errstate(invalid="ignore", over="ignore"):
        return M - (y_dst[None, :] - y_src[:, None])


class Ref:
    """Summary of one pass over the rows [row0, row0 + S_loc) of an S x D matrix, arc id (row0 + i) * D + j.
    count = #(rc < -tol) (NaN never violates); min = NaN-skipping minimum, +inf without a non-NaN arc, +0.0 for a
    zero minimum; nan = any rc is NaN; top-K = the violators by (rc, id), from a stable argsort."""

    def __init__(self, rc, row0, tol=TOL):
        self.rc = rc
        self.row0 = int(row0)
        self.D = rc.shape[1]
        flat = rc.ravel()
        with np.errstate(invalid="ignore"):
            viol = np.flatnonzero(flat < -tol)
        self.order = viol[np.argsort(flat[viol], kind="stable")]      # flat index ascending = id ascending
        mn = float(np.fmin.reduce(flat, initial=INF))
        self.min = 0.0 if mn == 0 else mn
        self.nan = bool(np.isnan(flat).any())

    @property
    def count(self):
        return int(self.order.size)

    def topk(self, K):
        o = self.order[:K]
        return (self.row0 * self.D + o).astype(np.int64), self.rc.ravel()[o]

    def k_cut(self, T):
        """(#violators below T, #arcs exactly at T)."""
        v = self.rc.ravel()[self.order]
        return int((v < T).sum()), int((v == T).sum())


def f64_bytes(v):
    return np.float64(v).tobytes()


def same_bits(got, ref):
    """NaN at the same positions and every other element bit for bit."""
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    assert got.shape == ref.shape
    gn, rn = np.isnan(got), np.isnan(ref)
    assert np.array_equal(gn, rn), f"NaN at {np.flatnonzero(gn != rn)[:10]}"
    bad = np.flatnonzero(got[~gn].view(np.uint64) != ref[~rn].view(np.uint64))
    assert bad.size == 0, f"{bad.size} elements differ, first at {np.flatnonzero(~gn)[bad[:5]]}: " \
                          f"{got[~gn][bad[:5]]} vs {ref[~rn][bad[:5]]}"


# ==== instances ============================================================================================
def row0_past_2p31(S_loc, D):
    """A first row whose slab has arc ids on both sides of 2^31."""
    return max(1, (1 << 31) // D - S_loc // 2)


TOL_VALUES = (-TOL, np.nextafter(-TOL, -INF), np.nextafter(-TOL, INF))   # at -tol, a violator, not a violator


def tol_duals(ys, yd, skip_rows):
    """Duals for rc = -tol and its two neighbours at three arcs (i_t, cols) of one row: there y_dst[j] == y_src[i],
    so the inner difference is exactly +0.0 and rc = M.  Duals move only so that no other reduced cost falls: the
    three sink duals drop to their smallest one b, the source dual of a row with y_src <= b rises to b."""
    S, D = ys.size, yd.size
    cols = sorted({j for j in (D - 2, D // 3 + 1, 1) if 0 <= j < D}) or [0]
    b = yd[cols].min()
    rows = [i for i in range(S) if i not in skip_rows and ys[i] <= b] or [i for i in range(S) if ys[i] <= b] or [S - 1]
    i_t = min(rows, key=lambda i: ys[i])
    yd[cols] = b
    ys[i_t] = b
    return i_t, cols


def plant_tol(M, i_t, cols):
    for j, v in zip(cols, TOL_VALUES):
        M[i_t, j] = v


def plant_ties(M, ys, yd, T, rows, cols):
    """M = T + w at (rows x cols) wherever fl(fl(T + w) - w) == T; returns the number of arcs planted."""
    w = yd[None, cols] - ys[rows, None]
    m = T + w
    ok = (m - w) == T
    sub = M[np.ix_(rows, cols)]
    sub[ok] = m[ok]
    M[np.ix_(rows, cols)] = sub
    return int(ok.sum())


def plant_special(M, ys, yd, R, rng, inf_violators):
    """NaN / +-inf costs and duals.  One NaN cost in the last row and last column of a tile (row R - 1, column
    255) and one at the last arc of the slab; one +inf and one -inf cost; a NaN, a +inf source dual and a -inf
    sink dual.  With inf_violators also a -inf source dual and a +inf sink dual, whose row / column is all -inf."""
    S, D = M.shape
    M[min(R, S) - 1, min(BOX_COLS, D) - 1] = NAN
    M[S - 1, D - 1] = NAN
    M[rng.integers(S), rng.integers(D)] = INF
    M[rng.integers(S), rng.integers(D)] = -INF
    rows = rng.permutation(S)
    cols = rng.permutation(D)
    ys[rows[0]] = NAN
    if S > 1:
        ys[rows[1]] = INF
    yd[cols[0]] = -INF
    if inf_violators:
        if S > 2:
            ys[rows[2]] = -INF
        if D > 1:
            yd[cols[1]] = INF


T_GRID = -0.25                # tie value of the small matrices: below the rc = -tol arcs, above the scattered violators


@functools.lru_cache(maxsize=None)
def grid_case(R, S_loc, D, special, seed=0):
    """(M, y_src, y_dst, row0, K) for an S_loc x D slab priced at box height R.  Sink duals in [3, 4), source duals
    in [0, 1): w = y_dst - y_src lies in (2, 4], where M = T + w is exact and M - w = T.  Base reduced costs are
    0.25 + U[0, 1) (no violator), up to 300 scattered violators in [-1, -0.5), a tie run at T_GRID over every row of
    the first two tiles at three columns (first, middle, last) and at a few random arcs, and the -tol arcs.
    K cuts the tie run in half."""
    rng = np.random.default_rng([seed, R, S_loc, D, int(special)])
    ys = rng.random(S_loc)
    yd = 3.0 + rng.random(D)
    tie_rows = list(range(min(S_loc, 2 * R)))
    i_t, tol_cols = tol_duals(ys, yd, set(tie_rows) if S_loc > 2 * R else set())
    M = (yd[None, :] - ys[:, None]) + (0.25 + rng.random((S_loc, D)))
    n = min(S_loc * D // 500, 300) + 1
    at = rng.choice(S_loc * D, n, replace=False)
    r, c = np.divmod(at, D)
    M[r, c] = (yd[c] - ys[r]) - (0.5 + 0.5 * rng.random(n))
    tie_cols = sorted({0, D // 2, D - 1} - set(tol_cols)) or [0]
    plant_ties(M, ys, yd, T_GRID, np.array(tie_rows), np.array(tie_cols))
    extra = rng.choice(S_loc * D, min(12, S_loc * D), replace=False)
    er, ec = np.divmod(extra, D)
    for i, j in zip(er, ec):
        plant_ties(M, ys, yd, T_GRID, np.array([i]), np.array([j]))
    plant_tol(M, i_t, tol_cols)
    if special:
        plant_special(M, ys, yd, R, rng, inf_violators=True)
    row0 = row0_past_2p31(S_loc, D)
    ref = Ref(rc_ref(M, ys, yd), row0)
    n_lt, n_eq = ref.k_cut(T_GRID)
    K = int(np.clip(n_lt + max(n_eq // 2, 1), 1, 1024))
    return M, ys, yd, row0, K, ref


def long_case(special):
    """6000 x 4099 with planted duals (noise 2e-3: ~0.05 % of the arcs violate), a tie run at the K = 1024 cut over
    rows 0 - 119 at columns 5, 1000 and 4098 (column blocks 0, 3 and the partial last one), the -tol arcs, and in
    the special flavour NaN / +inf costs and duals whose reduced costs are not violators (so the cut stays in the
    run), a -inf cost and NaN in the last row of a tile of every box height."""
    s, d, M = cases.ot_points(LONG_S, LONG_D, 20261022)
    y = cases.planted_duals(M, 20261022, 2e-3)
    ys, yd = y[:LONG_S].copy(), y[LONG_S:].copy()
    M = M.copy()
    tie_rows = np.arange(TIE_ROWS_LONG)
    tie_cols = np.array([5, 1000, LONG_D - 1])
    i_t, tol_cols = tol_duals(ys, yd, set(range(TIE_ROWS_LONG)))
    plant_tol(M, i_t, tol_cols)
    base = Ref(rc_ref(M, ys, yd), 0)
    v = base.rc.ravel()[base.order]
    T = float(np.floor(v[874] * 2.0 ** 24) / 2.0 ** 24)
    plant_ties(M, ys, yd, T, tie_rows, tie_cols)
    if special:
        rng = np.random.default_rng(7)
        plant_special(M, ys, yd, 16, rng, inf_violators=False)
        M[ROW_ALL_TILES, BOX_COLS - 1] = NAN
        M[ROW_ALL_TILES, LONG_D - 1] = NAN
    row0 = row0_past_2p31(LONG_S, LONG_D)
    ref = Ref(rc_ref(M, ys, yd), row0)
    n_lt, n_eq = ref.k_cut(T)
    assert n_lt < 1024 < n_lt + n_eq, (n_lt, n_eq)
    assert np.array_equal(ref.rc[i_t, tol_cols], TOL_VALUES)
    return M, ys, yd, row0, ref


# ==== CPU: the reference, the generator and the setters ====================================================
@pytest.mark.parametrize("name", OT_FULL)
def test_reference_reproduces_golden_reduced_costs(name):
    """rc_tree / rc_pert of the reference run byte for byte, its optimality flags, and the oracle's summary; the
    same summary from row slabs with row0 > 0."""
    fx = Fixture(name)
    M = fx.inp["M"]
    S, D = M.shape
    for tag in ("tree", "pert"):
        y = fx.out["y_" + tag]
        rc = rc_ref(M, y[:S], y[S:])
        assert rc.ravel().tobytes() == fx.out["rc_" + tag].tobytes()
        ref = Ref(rc, 0)
        assert (ref.count == 0 and not ref.nan) == bool(fx.out["optimal_" + tag])
        cnt, mn, ids, vals = orc.price_summary(fx.out["rc_" + tag], K=32)
        got_ids, got_vals = ref.topk(32)
        assert (ref.count, f64_bytes(ref.min)) == (cnt, f64_bytes(mn))
        assert np.array_equal(got_ids, ids) and got_vals.tobytes() == vals.tobytes()
        slabs = [Ref(rc_ref(M[r:r + 7], y[r:min(r + 7, S)], y[S:]), r) for r in range(0, S, 7)]
        assert sum(sl.count for sl in slabs) == cnt
        assert min(sl.min for sl in slabs) == mn
        merged = np.concatenate([sl.topk(32)[0] for sl in slabs])
        mvals = np.concatenate([sl.topk(32)[1] for sl in slabs])
        o = np.lexsort((merged, mvals))[:32]
        assert np.array_equal(merged[o], ids) and mvals[o].tobytes() == vals.tobytes()


def test_reference_reproduces_c2_summary():
    s, d, M, x = c2_inputs()
    small = Fixture("ot_c2_784_small").out
    S = M.shape[0]
    y = small["y_pert"]
    ref = Ref(rc_ref(M, y[:S], y[S:]), 0)
    assert cases.digest(ref.rc.ravel()) == digests()["ot_c2_784"]["digests"]["rc_pert"]
    assert ref.count == int(small["count_pert"]) and f64_bytes(ref.min) == f64_bytes(small["min_rc_pert"])
    assert np.array_equal(ref.topk(256)[0], small["topk_ids_pert"])


def test_reference_min_conventions():
    """+inf when every reduced cost is NaN, +0.0 for a zero minimum, NaN never a violator."""
    r = Ref(np.full((2, 3), NAN), 5)
    assert r.min == INF and r.count == 0 and r.nan
    r = Ref(np.array([[-0.0, 1.0], [NAN, 0.0]]), 0)
    assert f64_bytes(r.min) == f64_bytes(0.0) and r.count == 0 and r.nan
    r = Ref(np.array([[-TOL, np.nextafter(-TOL, -INF), -INF]]), 1)
    assert r.count == 2 and r.min == -INF and np.array_equal(r.topk(5)[0], [5, 4])


@pytest.mark.parametrize("special", [False, True])
def test_generator_plants_what_it_claims(special):
    """A 56 x 1001 slab at box height 16: ids straddle 2^31, K cuts the tie run, -tol and its neighbours, the tie
    run covers all rows of the first two tiles, NaN at a tile's last row and column."""
    R, S_loc, D = 16, 56, 1001
    M, ys, yd, row0, K, ref = grid_case(R, S_loc, D, special)
    assert row0 * D < (1 << 31) < (row0 + S_loc) * D
    rc = ref.rc
    n_lt, n_eq = ref.k_cut(T_GRID)
    assert n_eq >= 2 * R * 3 - 3 and K > 1
    assert min((rc == v).sum() for v in TOL_VALUES) >= 1
    if special:
        assert np.isnan(rc[R - 1, BOX_COLS - 1]) and np.isnan(rc[-1, -1]) and ref.nan
        assert np.isneginf(rc).sum() >= S_loc + D - 6 and np.isposinf(rc).any()
    else:
        assert n_lt < K < n_lt + n_eq and np.all(rc[:2 * R, [0, D // 2, D - 1]] == T_GRID)
        assert not ref.nan and np.isfinite(rc).all() and ref.min < -0.5


def test_setters_reject_out_of_range(lib):
    assert lib.sx_price_set_tuning(len(TMA_SHAPES), 0) == ERR_INVALID
    assert lib.sx_price_set_tma_options(4, -1) == ERR_INVALID
    assert lib.sx_score_set_tuning(2) == ERR_INVALID
    assert lib.sx_score_set_tuning(5) == ERR_INVALID
    for q in range(len(TMA_SHAPES)):
        assert lib.sx_price_set_tuning(q, 0) == 0
    assert lib.sx_price_set_tma_options(0, 0) == 0
    assert lib.sx_score_set_tuning(3) == 0


# ==== fixtures =============================================================================================
def restore_defaults(lib):
    assert lib.sx_price_set_tuning(DEFAULT_SHAPE, DEFAULT_DIRECT_CTAS) == 0
    assert lib.sx_price_set_tma_options(DEFAULT_L2, DEFAULT_EVICT) == 0
    assert lib.sx_score_set_tuning(DEFAULT_SCORE_CTAS) == 0


@pytest.fixture
def lib():
    """The native library with its tuning restored to the defaults afterwards, whatever the test did."""
    from smart_crossover._native import lib as native
    try:
        yield native
    finally:
        restore_defaults(native)


@pytest.fixture(scope="module")
def dev():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from smart_crossover import device
    return device


@pytest.fixture
def knobs(dev, lib):
    """`lib` for a GPU test: skipped without a device, tuning restored afterwards."""
    return lib


def num_sms():
    import torch
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _vp(t, byte_offset=0):
    return ctypes.c_void_p(t.data_ptr() + byte_offset)


class Slab:
    """M as rows 1 .. S_loc of a NaN-filled (S_loc + 2) x ld device buffer, starting `col` elements into the row
    (col = 1: an 8-byte offset base), with y_src / y_dst on the device."""

    def __init__(self, M, ys, yd, ld, col=0):
        import torch
        S, D = M.shape
        assert ld >= D + col
        self.buf = torch.full((S + 2, ld), NAN, dtype=torch.float64, device="cuda")
        self.buf[1:S + 1, col:col + D] = torch.from_numpy(M).cuda()
        self.ys = torch.from_numpy(np.ascontiguousarray(ys)).cuda()
        self.yd = torch.from_numpy(np.ascontiguousarray(yd)).cuda()
        self.S, self.D, self.ld, self.col = S, D, ld, col

    @property
    def ptr(self):
        return _vp(self.buf[1], 8 * self.col)


class RcOut:
    """rc_out as rows 1 .. S_loc of a SENTINEL-filled (S_loc + 2) x ld_out buffer, ld_out > D."""

    def __init__(self, S, D, ld_out):
        import torch
        self.buf = torch.full((S + 2, ld_out), SENTINEL, dtype=torch.float64, device="cuda")
        self.S, self.D, self.ld_out = S, D, ld_out

    def check(self, ref_dev):
        import torch
        body = self.buf[1:self.S + 1, :self.D]
        gn, rn = torch.isnan(body), torch.isnan(ref_dev)
        assert torch.equal(gn, rn), "NaN reduced costs at other arcs"
        bad = (body.view(torch.int64) != ref_dev.view(torch.int64)) & ~gn
        if bad.any():
            i, j = (int(v) for v in bad.nonzero()[0])
            raise AssertionError(f"{int(bad.sum())} reduced costs differ, first at ({i}, {j}): "
                                 f"{float(body[i, j])!r} vs {float(ref_dev[i, j])!r}")
        sent = torch.tensor([SENTINEL], dtype=torch.float64, device="cuda").view(torch.int64)
        pad = torch.cat([self.buf[0], self.buf[self.S + 1], self.buf[1:self.S + 1, self.D:].reshape(-1)])
        assert torch.equal(pad.view(torch.int64), sent.expand(pad.numel())), "rc_out written outside the slab"


def price(dev, slab, row0, K, rc_out=None, variant=0, cand_cap=None):
    """One pass through lib.sx_price_dense_ot (begin, price, select, fetch), repeated after a candidate overflow
    with a grown buffer.  Returns (result, n_priced of the last pass, number of repeats)."""
    import torch
    from smart_crossover._native import check, lib
    pr = dev.Pricer(torch.device("cuda"), K, cand_cap=cand_cap, fused=False)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    repeats = 0
    while True:
        pr.reset()
        check(lib.sx_price_dense_ot(slab.ptr, slab.ld, row0, slab.S, slab.D, _vp(slab.ys), _vp(slab.yd), TOL,
                                    _vp(pr.header), _vp(pr.sel), _vp(pr.cand_rc), _vp(pr.cand_id), pr.cap,
                                    _vp(rc_out.buf[1]) if rc_out is not None else None,
                                    rc_out.ld_out if rc_out is not None else 0, variant, stream), "sx_price_dense_ot")
        pr.select()
        res = pr.fetch()
        if not pr.overflowed(res):
            return res, int(pr.h_block[2 * pr.Kp + 2]), repeats
        repeats += 1
        pr.grow(res.n_violating)


def check_pass(res, n_priced, ref, K, what=""):
    ids, vals = ref.topk(K)
    assert res.n_violating == ref.count, what
    assert f64_bytes(res.min_rc) == f64_bytes(ref.min), f"{what}: min {res.min_rc!r} vs {ref.min!r}"
    assert res.topk_id.size == ids.size, f"{what}: {res.topk_id.size} of {ids.size} selected"
    assert np.array_equal(res.topk_id, ids), f"{what}: top-{K} ids differ at {np.flatnonzero(res.topk_id != ids)[:8]}"
    assert res.topk_rc.tobytes() == vals.tobytes(), what
    assert res.status == (NAN_RC if ref.nan else 0), what
    assert n_priced == ref.rc.size, what


def even_ld(D, extra=0):
    """The smallest even leading dimension > D + extra."""
    ld = D + extra + 1
    return ld + (ld & 1)


def to_dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ==== GPU: every TMA shape on the boundary grid ============================================================
@pytest.mark.gpu
@pytest.mark.parametrize("write_rc", [False, True], ids=["count", "rc_out"])
@pytest.mark.parametrize("shape", range(len(TMA_SHAPES)))
def test_tma_shape_boundary_grid(knobs, dev, shape, write_rc):
    """S_loc in {1, R - 1, R, R + 1, 3R + R/2} x D in {1, 2, 255, 256, 257, 512, 1001}, finite and special content,
    K at the middle of the tie run and K = 1."""
    R = TMA_SHAPES[shape][0]
    assert knobs.sx_price_set_tuning(shape, 0) == 0
    for S_loc in (1, R - 1, R, R + 1, 3 * R + R // 2):
        for D in GRID_D:
            for special in (False, True):
                M, ys, yd, row0, K, ref = grid_case(R, S_loc, D, special)
                slab = Slab(M, ys, yd, even_ld(D))
                out = RcOut(S_loc, D, D + 3) if write_rc else None
                what = f"shape {shape} S_loc {S_loc} D {D} special {special}"
                for k in (K, 1):
                    res, n_priced, _ = price(dev, slab, row0, k, rc_out=out)
                    check_pass(res, n_priced, ref, k, f"{what} K {k}")
                if write_rc:
                    out.check(to_dev(ref.rc))


# ==== GPU: every TMA shape on the long matrix ==============================================================
@pytest.fixture(scope="module")
def long_mats(dev):
    """Both flavours of the long matrix, on the device with their reference reduced costs."""
    out = {}
    for special in (False, True):
        M, ys, yd, row0, ref = long_case(special)
        out[special] = (Slab(M, ys, yd, LONG_LD), row0, ref, to_dev(ref.rc))
    return out


def ring_wraps(shape):
    rows, stages, _, ctas = TMA_SHAPES[shape]
    tiles = -(-LONG_S // rows) * -(-LONG_D // BOX_COLS)
    return tiles // (num_sms() * ctas) // stages


@pytest.mark.gpu
@pytest.mark.parametrize("write_rc", [False, True], ids=["count", "rc_out"])
@pytest.mark.parametrize("shape", range(len(TMA_SHAPES)))
def test_tma_shape_long_walk(knobs, dev, long_mats, shape, write_rc):
    """Every CTA wraps its ring >= 4 times.  K = 1 and K = 1024 (which cuts the tie run) on both flavours, and the
    candidate-overflow repeat from a 64-entry candidate buffer."""
    assert ring_wraps(shape) >= 4, f"shape {shape}: the long matrix is too small for this device"
    assert knobs.sx_price_set_tuning(shape, 0) == 0
    for special in (False, True):
        slab, row0, ref, ref_dev = long_mats[special]
        out = RcOut(LONG_S, LONG_D, LONG_D + 5) if write_rc else None
        for K in (1, 1024):
            res, n_priced, repeats = price(dev, slab, row0, K, rc_out=out if K == 1 else None)
            check_pass(res, n_priced, ref, K, f"shape {shape} special {special} K {K}")
            assert repeats == 0
        if write_rc:
            out.check(ref_dev)
    slab, row0, ref, _ = long_mats[False]
    res, n_priced, repeats = price(dev, slab, row0, 1024, cand_cap=64)
    assert repeats >= 1
    check_pass(res, n_priced, ref, 1024, f"shape {shape} after {repeats} overflow repeats")


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [6, 8])
def test_tma_cache_hints_change_nothing(knobs, dev, long_mats, shape):
    """L2 promotion 0 - 3 x evict-first 0 / 1 are cache hints: the same bits at shape 6 and at shape 8
    (16 consumer warps, 6 rows per thread)."""
    assert knobs.sx_price_set_tuning(shape, 0) == 0
    slab, row0, ref, ref_dev = long_mats[True]
    for l2 in range(4):
        for evict in (0, 1):
            assert knobs.sx_price_set_tma_options(l2, evict) == 0
            out = RcOut(LONG_S, LONG_D, LONG_D + 1)
            res, n_priced, _ = price(dev, slab, row0, 1024, rc_out=out)
            check_pass(res, n_priced, ref, 1024, f"shape {shape} l2 {l2} evict {evict}")
            out.check(ref_dev)


# ==== GPU: the direct-load kernels =========================================================================
def direct_shapes(G):
    """(relation, S_loc, D) such that the grid G (when the tiles outnumber it) is smaller than, equal to, a
    multiple of, and k * n_col_blocks + r with 0 < r < n_col_blocks."""
    q = next(p for p in range(2, G + 1) if G % p == 0)
    ncb3 = G // 3 + 1
    k, r = divmod(G, ncb3)
    assert k >= 1 and 0 < r < ncb3
    return [("G < ncb", 3, BOX_COLS * (G + 3) - 5),
            ("G = ncb", 3 * DIRECT_ROWS + 5, BOX_COLS * G - 7),
            (f"G = {q} ncb", DIRECT_ROWS * (q + 2) + 3, BOX_COLS * (G // q) - 1),
            (f"G = {k} ncb + {r}", DIRECT_ROWS * (k + 2) + 5, BOX_COLS * ncb3 - 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("ctas", [1, 3, 4, 8, 16, 40])
def test_direct_variants_grid_walk(knobs, dev, ctas):
    """Variant 1 on an aligned slab, variant 2 on one whose base is 8 bytes past a 16-byte boundary (variants 0
    and 1 reject it), each with and without rc_out."""
    assert knobs.sx_price_set_tuning(-1, ctas) == 0
    G = num_sms() * ctas
    for n, (rel, S_loc, D) in enumerate(direct_shapes(G)):
        ncb = -(-D // BOX_COLS)
        assert -(-S_loc // DIRECT_ROWS) * ncb > G, rel
        special = bool(n & 1)
        M, ys, yd, row0, K, ref = grid_case.__wrapped__(DIRECT_ROWS, S_loc, D, special, seed=ctas)   # not cached
        ref_dev = to_dev(ref.rc)
        for variant, col in ((1, 0), (2, 1)):
            slab = Slab(M, ys, yd, even_ld(D, col), col)
            what = f"{ctas} CTAs/SM, {rel}, S_loc {S_loc} D {D}, variant {variant}"
            if col:
                for v in (0, 1):
                    with pytest.raises(dev._native.SxError) as e:
                        price(dev, slab, row0, K, variant=v)
                    assert e.value.code == ERR_UNALIGNED
            out = RcOut(S_loc, D, D + 1)
            res, n_priced, _ = price(dev, slab, row0, K, rc_out=out, variant=variant)
            check_pass(res, n_priced, ref, K, what + " rc_out")
            out.check(ref_dev)
            res, n_priced, _ = price(dev, slab, row0, K, variant=variant)
            check_pass(res, n_priced, ref, K, what)
        del slab, out, ref_dev


# ==== GPU: the score kernel at 3 and 4 CTAs per SM =========================================================
def score_ref(x, s, d):
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        return np.maximum(x.reshape(s.size, d.size) / s[:, None], x.reshape(s.size, d.size) / d[None, :]).ravel()


def hist12_ref(v):
    """np.bincount of the top 12 bits of the order-preserving key: -0.0 -> +0.0, NaN -> all ones, negative ->
    ~bits, else bits | 1 << 63."""
    b = np.asarray(v, dtype=np.float64).view(np.uint64).copy()
    b[(b << np.uint64(1)) == 0] = 0
    neg = (b >> np.uint64(63)) == 1
    key = np.where(neg, ~b, b | np.uint64(1 << 63))
    key[np.isnan(v)] = np.uint64(0xFFFFFFFFFFFFFFFF)
    return np.bincount((key >> np.uint64(52)).astype(np.int64), minlength=4096)


def score_inputs(S, D, seed):
    """Positive flows and marginals with negative x, -0.0, +0.0, NaN, +-inf, subnormal and huge x, and zero
    marginals (x / 0 = +-inf, 0 / 0 = NaN)."""
    rng = np.random.default_rng(seed)
    s = rng.random(S) + 1e-3
    d = rng.random(D) + 1e-3
    x = rng.random(S * D) * 1e-3
    specials = np.array([-1.5, -0.0, 0.0, NAN, INF, -INF, 5e-324, 1e308, -3e-300, 2.0 ** -1022])
    at = rng.choice(S * D, min(S * D, 4000), replace=False)
    x[at] = specials[np.arange(at.size) % specials.size]
    s[rng.choice(S, max(1, S // 50), replace=False)] = 0.0
    d[rng.choice(D, max(1, D // 50), replace=False)] = 0.0
    return x, s, d


@pytest.mark.gpu
@pytest.mark.parametrize("score_ctas", [3, 4])
@pytest.mark.parametrize("S,D", [(1, 2), (37, 2050), (1000, 4106), (5, 3), (300, 4105)],
                         ids=["1x2", "37x2050", "1000x4106", "5x3-odd", "300x4105-odd"])
def test_score_tuning_scores_and_histogram(knobs, dev, score_ctas, S, D):
    """Even D takes score_ot_vec_kernel<HIST, score_ctas> (with and without the histogram); odd D the scalar
    kernel + sx_hist12_f64.  Scores bit for bit (NaN by position), the histogram exactly."""
    assert knobs.sx_score_set_tuning(score_ctas) == 0
    x, s, d = score_inputs(S, D, 1000 * S + D)
    ref = score_ref(x, s, d)
    if S * D > 1000:
        assert np.isnan(ref).any() and np.isposinf(ref).any() and np.isneginf(ref).any() and (ref < 0).any()
    hist_ref = hist12_ref(ref)
    out, hist = dev.score_ot(to_dev(x), to_dev(s), to_dev(d), want_hist=True)
    same_bits(out.cpu().numpy(), ref)
    assert np.array_equal(hist.cpu().numpy().astype(np.int64), hist_ref)
    same_bits(dev.score_ot(to_dev(x), to_dev(s), to_dev(d)).cpu().numpy(), ref)

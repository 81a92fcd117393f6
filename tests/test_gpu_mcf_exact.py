"""The min-cost-flow kernels against literal NumPy / SciPy references.

sx_score_mcf gives the flow indicators of `MCFManagerStd.get_sorted_flows`; sx_price_arcs prices an arc list for
`MCFManagerStd.price`.  Both are bit-exact by contract, so every GPU assertion here compares bytes: NaN positions
first, then the bytes of everything else.  No tolerance is used anywhere.

  * Scores.  `mcf_scores_ref` writes net_manager.py:165-182 out in NumPy / SciPy, independently of the oracle's C
    loop: the reversal mask, x_hat, the flipped incidence matrix split into a CSR matrix of its +1 entries and one of
    its negated -1 entries, whose `@` is SciPy's csr_matvec (per node, a sequential sum from 0.0 in ascending arc
    id), f_inv = 1 / max(f1, f2) or 0, and per arc the NumPy maximum over its two end nodes of |f_inv * x_hat|.
    Cases: every branch of the reversal and zeroing rule, nodes with f1 > f2, f1 < f2, f1 == f2, f == 0, f == inf
    and f_inv == inf, isolated nodes and parallel arcs; a hub of degree > 2^17 whose scores change under any other
    summation order; node and arc counts at the kernels' grid-stride sweeps; and the manager with A stored in four
    forms.
  * Pricing.  rc = c - (y[tail] - y[head]), negated where vbasis == -2, summarised by `summary_ref`.  Cases: NaN and
    infinite costs and duals, the sign of zero under the negation, rc == -tol on both kernels, every alignment
    (vector bulk + scalar tail, everything scalar), ids past 2^31, one pass accumulated from three calls,
    K = 1 / 1024 / 3000 on tied costs, the candidate-overflow repeat, and the manager after its big-M extension.

Where the reference's own code leaves a point open, these tests pin the kernels' behaviour (include/sxcross.h says
the same next to the entry points):
  * A stored zero in the incidence matrix is not an incidence.  It enters neither node sum, so a NaN or infinite
    x_hat of that arc cannot make the node's sum NaN through it.
  * min_rc is the minimum over the reduced costs that are not NaN, +inf when every one is NaN (as for an empty
    list).  A zero minimum is reported as +0.0.

The tests without the `gpu` marker check the references themselves: against the golden scores of the reference
run, against the oracle on the C3 generator, and, as a negative control, that summing the hub instance's node
sums in another order changes their bits and the hub arcs' scores.
"""
import numpy as np
import pytest
import scipy.sparse as sp

import cases
from golden_util import MCF_FULL, Fixture
from oracle import network_oracle as orc

TOL = 1e-6                    # TOLERANCE_FOR_REDUCED_COSTS
DBL_MAX = np.finfo(np.float64).max
TINY = np.nextafter(0.0, 1.0)  # smallest subnormal
INF, NAN = np.inf, np.nan
NAN_RC = 8                    # SX_STATUS_NAN_RC
ID0_FAR = 3_000_000_000       # arc ids offset past 2^31


# ==== references ===========================================================================================
def incidence(tail, head, N):
    """N x E node-arc incidence matrix, +1 at the tail and -1 at the head, canonical CSR."""
    E = tail.size
    A = sp.csr_matrix((np.concatenate([np.ones(E), -np.ones(E)]),
                       (np.concatenate([tail, head]), np.concatenate([np.arange(E)] * 2))), shape=(N, E))
    A.sort_indices()
    return A


def xhat_ref(x, u):
    """net_manager.py:166-169 as written: (x_hat, mask)."""
    with np.errstate(invalid="ignore", over="ignore"):
        mask = x > u / 2
        x_hat = x * (~mask) + u * mask - x * mask
        x_hat[(x < 0) | (x > u)] = 0
    return x_hat, mask


def flipped_parts(A, mask):
    """A_bar (A with the columns of reversed arcs negated) as two CSR matrices with sorted indices: its +1 entries
    and its negated -1 entries.  Stored zeros of A are dropped: they are no incidence."""
    A = sp.csr_matrix(A, copy=True)
    A.sort_indices()
    d = np.where(mask[A.indices], -A.data, A.data)
    parts = []
    for vals in (np.where(d > 0, d, 0.0), np.where(d < 0, -d, 0.0)):
        P = sp.csr_matrix((vals, A.indices.copy(), A.indptr.copy()), shape=A.shape)
        P.eliminate_zeros()
        assert P.has_sorted_indices
        parts.append(P)
    return parts


def node_sums_ref(A, x_hat, mask):
    """f1 = A_bar+ @ x_hat, f2 = A_bar- @ x_hat (csr_matvec: sequential from 0.0 in ascending arc id)."""
    pos, neg = flipped_parts(A, mask)
    with np.errstate(invalid="ignore", over="ignore"):
        return pos @ x_hat, neg @ x_hat


def scores_from_sums(f1, f2, x_hat, tail, head):
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        f = np.maximum(f1, f2)
        f_inv = np.divide(1.0, f, out=np.zeros_like(f), where=f != 0)
        return np.maximum(np.maximum(0.0, np.abs(f_inv[tail] * x_hat)), np.abs(f_inv[head] * x_hat))


def mcf_scores_ref(x, u, A, tail, head):
    x = np.asarray(x, dtype=np.float64)
    u = np.asarray(u, dtype=np.float64)
    x_hat, mask = xhat_ref(x, u)
    f1, f2 = node_sums_ref(A, x_hat, mask)
    return scores_from_sums(f1, f2, x_hat, tail, head)


def rc_ref(c, tail, head, y, vbasis=None):
    """net_manager.py:302-303: rc = c - (y_tail - y_head), negated where vbasis == -2."""
    with np.errstate(invalid="ignore"):
        rc = c - (y[tail] - y[head])
    if vbasis is not None:
        flip = np.asarray(vbasis) == -2
        rc[flip] = -rc[flip]
    return rc


def summary_ref(rc, K, tol=TOL):
    """(count, min, top-K ids, top-K rc, any NaN) with `price_summary` semantics: violators are rc < -tol, ranked by
    (rc, id) ascending; NaN is never counted or selected.  The minimum skips NaN (+inf if nothing else is left); a
    zero minimum is +0.0."""
    with np.errstate(invalid="ignore"):
        viol = np.flatnonzero(rc < -tol)
    ok = rc[~np.isnan(rc)]
    mn = float(ok.min()) if ok.size else INF
    if mn == 0:
        mn = 0.0
    o = viol[np.argsort(rc[viol], kind="stable")][:K]
    return int(viol.size), mn, o.astype(np.int64), rc[o], bool(np.isnan(rc).any())


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
def branch_pairs():
    """(x, u) pairs that reach every branch of the reversal / zeroing rule."""
    six = 6.0
    return [
        (3.0, six),                              # x == u/2: not reversed
        (np.nextafter(3.0, INF), six),           # just above: reversed
        (np.nextafter(3.0, -INF), six),          # just below
        (six, six),                              # x == u: reversed, x_hat = 0
        (np.nextafter(six, INF), six),           # x > u: zeroed
        (2 * six, six),                          # x = 2u: zeroed
        (-1.0, six),                             # x < 0: zeroed
        (-0.0, six), (0.0, six),
        (0.0, 0.0), (1.0, 0.0),                  # u == 0
        (0.0, TINY), (TINY, TINY),               # u/2 rounds to 0
        (DBL_MAX, DBL_MAX), (np.nextafter(DBL_MAX, 0), DBL_MAX), (DBL_MAX / 2, DBL_MAX),
        (0.75 * DBL_MAX, DBL_MAX), (0.4 * DBL_MAX, DBL_MAX),
        (NAN, six), (5.0, NAN),
        (1.0, INF), (0.0, INF), (INF, INF),      # u == inf: x_hat = x + inf * 0 = NaN
        (1.0, -2.0),                             # negative capacity: reversed, then zeroed
        (TINY, 1.0),                             # a lone subnormal x_hat: f = TINY, f_inv = inf
    ]


def branch_instance(seed, with_nan=True):
    """Ring plus chords with parallel and antiparallel arcs, isolated nodes (in the middle and at the end), the
    branch pairs spread over the arcs (each used twice) and small integer flows elsewhere, so that f1 == f2 occurs.
    Returns (tail, head, x, u, N)."""
    rng = np.random.default_rng(seed)
    iso = {7, 40}
    N = 102
    ring = np.array([v for v in range(N - 5) if v not in iso])             # N-3 .. N-1 isolated as well
    t = list(ring)
    h = list(np.roll(ring, -1))
    flip = rng.random(len(t)) < 0.3                                        # some ring arcs point backwards
    t, h = np.where(flip, h, t), np.where(flip, t, h)
    n_chord = 160
    ct = rng.choice(ring, n_chord)
    ch = rng.choice(ring, n_chord)
    keep = ct != ch
    ct, ch = ct[keep], ch[keep]
    tail = np.concatenate([t, ct, ct[:6], ch[6:10]])                       # parallel and antiparallel copies
    head = np.concatenate([h, ch, ch[:6], ct[6:10]])
    perm = rng.permutation(tail.size)
    tail, head = tail[perm].astype(np.int64), head[perm].astype(np.int64)
    E = tail.size
    u = rng.integers(4, 12, E).astype(np.float64)
    x = rng.integers(0, 3, E).astype(np.float64)                           # x <= u/2: x_hat = x, small integers
    pairs = [p for p in branch_pairs() if with_nan or not np.isnan(xhat_ref(np.array([p[0]]), np.array([p[1]]))[0][0])]
    at = rng.choice(E, 2 * len(pairs), replace=False)
    for q, k in enumerate(at):
        x[k], u[k] = pairs[q % len(pairs)]
    # pendant nodes 97 and 98 whose arcs carry no flow: f == 0 there, f_inv = 0
    tail = np.concatenate([tail, [97, 0, 98]])
    head = np.concatenate([head, [1, 97, 2]])
    x = np.concatenate([x, [0.0, 0.0, 0.0]])
    u = np.concatenate([u, [5.0, 0.0, 3.0]])
    return tail, head, x, u, N


def special_nodes_instance():
    """Small hand-made nodes that the random instance may miss: f == inf (three arcs of 0.4 DBL_MAX), f_inv == inf
    next to an x_hat of 0 (inf * 0), f == 0 next to a node with f > 0, f1 == f2 exactly.  (tail, head, x, u, N)."""
    arcs = [  # (tail, head, x, u)
        (0, 1, 0.4 * DBL_MAX, DBL_MAX), (0, 2, 0.4 * DBL_MAX, DBL_MAX), (0, 3, 0.4 * DBL_MAX, DBL_MAX),
        (4, 5, TINY, 1.0), (5, 6, 0.0, 1.0), (7, 5, 0.0, 3.0),
        (8, 9, 0.0, 2.0), (9, 10, 2.0, 4.0),
        (11, 12, 1.5, 4.0), (12, 13, 1.5, 4.0), (13, 11, 2.5, 4.0),      # reversed: f1 > f2, ==, < round it
    ]
    t, h, x, u = (np.array(v) for v in zip(*arcs))
    return t.astype(np.int64), h.astype(np.int64), x.astype(np.float64), u.astype(np.float64), 15


def hub_instance(seed):
    """Hub node 0 with 2^17 + 5 arcs, four nodes of degree ~1000, x_hat spread over 1e-12 .. 1e6.  Their arcs end at
    two 'big' nodes whose own f is larger (each also carries arcs of x_hat 1e13 to leaves), so every hub / mid arc's
    score is x_hat / f at the hub or mid node and shows that node's sum.  Arc ids shuffled.  (tail, head, x, u, N)."""
    rng = np.random.default_rng(seed)
    hub, big, mid = 0, np.array([1, 2]), np.arange(3, 7)
    n_leaf = 40
    leaves = np.arange(7, 7 + n_leaf)
    N = 7 + n_leaf + 2                                                     # two isolated nodes at the end
    a_own = np.concatenate([np.full((1 << 17) + 5, hub), np.repeat(mid, rng.integers(950, 1050, mid.size))])
    a_oth = rng.choice(big, a_own.size)
    g_own, g_oth = np.repeat(big, n_leaf // 2), leaves
    own = np.concatenate([a_own, g_own])
    oth = np.concatenate([a_oth, g_oth])
    out = rng.random(own.size) < 0.5                                       # both directions at every node
    tail, head = np.where(out, own, oth), np.where(out, oth, own)
    E = tail.size
    target = 10.0 ** rng.uniform(-12, 6, E)
    target[a_own.size:] = 1e13
    u = 4 * target
    rev = rng.random(E) < 0.3                                              # reversed arcs: x_hat = u - x
    x = np.where(rev, 3 * target, target)
    perm = rng.permutation(E)
    return tail[perm].astype(np.int64), head[perm].astype(np.int64), x[perm], u[perm], N


def sweep_instance(N, E, seed):
    """NETGEN-like ring + random arcs with interior flows and a sprinkle of the branch pairs."""
    tail, head, b, c, u = cases.netgen_like(N, E, seed)
    x = cases.mcf_interior_flow(u, seed)
    rng = np.random.default_rng(seed)
    pairs = branch_pairs()
    at = rng.choice(E, 4 * len(pairs), replace=False)
    for q, k in enumerate(at):
        x[k], u[k] = pairs[q % len(pairs)]
    return tail, head, x, u


# ==== CPU: the references themselves =======================================================================
@pytest.mark.parametrize("name", MCF_FULL)
def test_reference_scores_equal_golden(name):
    fx = Fixture(name)
    tail, head, x, u = (fx.inp[k] for k in ("tail", "head", "x", "u"))
    A = incidence(tail, head, fx.inp["b"].size)
    got = mcf_scores_ref(x, u, A, tail, head)
    assert got.tobytes() == fx.out["scores"].tobytes()
    assert np.array_equal(np.argsort(got, kind="stable")[::-1], fx.out["queue"])


@pytest.mark.parametrize("N,E,seed", [(2000, 20000, 5), (5000, 40000, 20260003)])
def test_reference_scores_equal_oracle_on_c3_generator(N, E, seed):
    tail, head, b, c, u = cases.netgen_like(N, E, seed)
    x = cases.mcf_interior_flow(u, seed)
    A = incidence(tail, head, N)
    assert mcf_scores_ref(x, u, A, tail, head).tobytes() == orc.mcf_flow_scores(x, u, A).tobytes()


def test_reference_matches_oracle_off_the_nan_branches():
    """Away from NaN the oracle and the reference agree on the branch instance too (the oracle multiplies by the
    stored entry, which only matters for NaN)."""
    tail, head, x, u, N = branch_instance(1, with_nan=False)
    A = incidence(tail, head, N)
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        same_bits(mcf_scores_ref(x, u, A, tail, head), orc.mcf_flow_scores(x, u, A))


def test_branch_instance_covers_every_case():
    """The branch and special-node instances reach what the GPU tests claim they reach."""
    for inst in (branch_instance(1), special_nodes_instance()):
        tail, head, x, u, N = inst
        A = incidence(tail, head, N)
        x_hat, mask = xhat_ref(x, u)
        f1, f2 = node_sums_ref(A, x_hat, mask)
        deg = np.diff(A.indptr)
        live = deg > 0
        with np.errstate(invalid="ignore"):
            kinds = {"f1>f2": (f1 > f2) & live, "f1<f2": (f1 < f2) & live, "f1==f2>0": (f1 == f2) & (f1 > 0),
                     "f==0": (np.maximum(f1, f2) == 0) & live, "isolated": ~live}
        for kind, hit in kinds.items():
            assert hit.any(), kind
    tail, head, x, u, N = branch_instance(1)
    A = incidence(tail, head, N)
    x_hat, mask = xhat_ref(x, u)
    f1, f2 = node_sums_ref(A, x_hat, mask)
    assert np.isnan(x_hat).any() and np.isnan(f1 + f2).any()
    pairs = set(zip(np.minimum(tail, head).tolist(), np.maximum(tail, head).tolist()))
    assert len(pairs) < tail.size                                          # parallel arcs
    tail, head, x, u, N = special_nodes_instance()
    A = incidence(tail, head, N)
    x_hat, mask = xhat_ref(x, u)
    f1, f2 = node_sums_ref(A, x_hat, mask)
    assert np.isinf(np.maximum(f1, f2)).any()                              # f == inf: f_inv = 0
    assert (np.maximum(f1, f2) == TINY).any()                              # f_inv == inf
    sc = mcf_scores_ref(x, u, A, tail, head)
    assert np.isnan(sc).any() and np.isinf(sc).any()                       # inf * 0 and inf * TINY


def _sequential(terms):
    return np.cumsum(terms)[-1] if terms.size else 0.0


def test_hub_sums_are_order_sensitive():
    """Negative control for test_score_hub_summation_order: csr_matvec is the sequential ascending-id sum, and the
    hub's and the mid nodes' sums in descending id or in np.sum's pairwise order have other bits, and so do the
    scores of their arcs."""
    tail, head, x, u, N = hub_instance(11)
    A = incidence(tail, head, N)
    x_hat, mask = xhat_ref(x, u)
    parts = flipped_parts(A, mask)
    sums = [P @ x_hat for P in parts]
    alt = {"reversed": [s.copy() for s in sums], "pairwise": [s.copy() for s in sums]}
    for P, s, r, p in zip(parts, sums, alt["reversed"], alt["pairwise"]):
        for v in range(7):
            terms = P.data[P.indptr[v]:P.indptr[v + 1]] * x_hat[P.indices[P.indptr[v]:P.indptr[v + 1]]]
            assert _sequential(terms) == s[v]
            r[v] = _sequential(terms[::-1])
            p[v] = np.sum(terms)
    deg = np.diff(A.indptr)
    assert deg[0] >= 1 << 17 and np.all((deg[3:7] >= 900) & (deg[3:7] <= 1100))
    ref = scores_from_sums(sums[0], sums[1], x_hat, tail, head)
    own = np.isin(tail, [0, 3, 4, 5, 6]) | np.isin(head, [0, 3, 4, 5, 6])
    for name, (a1, a2) in alt.items():
        for v in [0, 3, 4, 5, 6]:
            assert (a1[v], a2[v]) != (sums[0][v], sums[1][v]), (name, v)
        assert a1[0] != sums[0][0] and a2[0] != sums[1][0], name
        changed = ref != scores_from_sums(a1, a2, x_hat, tail, head)
        assert changed[own].mean() > 0.5, name                             # most hub / mid arcs change bits
        hub_arcs = (tail == 0) | (head == 0)
        assert changed[hub_arcs].mean() > 0.5, name


# ==== GPU fixtures =========================================================================================
@pytest.fixture(scope="module")
def dev():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from smart_crossover import device
    return device


def cu(a, dtype=None):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda()


def num_sms():
    import torch
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def score_dev(dev, x, u, tail, head, A):
    import torch
    A = sp.csr_matrix(A)
    if not A.has_sorted_indices:
        A = A.sorted_indices()
    out = dev.score_mcf(cu(x), cu(u), cu(tail, torch.int32), cu(head, torch.int32), cu(A.indptr, torch.int64),
                        cu(A.indices, torch.int32), cu(np.sign(A.data), torch.int8))
    return out.cpu().numpy()


def check_scores(dev, tail, head, x, u, N):
    A = incidence(tail, head, N)
    ref = mcf_scores_ref(x, u, A, tail, head)
    same_bits(score_dev(dev, x, u, tail, head, A), ref)
    return ref


# ==== GPU: sx_score_mcf ====================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_score_every_branch(dev, seed):
    """x == u/2 and its neighbours, x == u, x > u, x < 0, -0.0, u == 0, subnormal u, DBL_MAX, NaN, u == inf, on a
    ring with chords, parallel arcs and isolated nodes; also without the NaN pairs, where NaN cannot hide a branch."""
    check_scores(dev, *branch_instance(seed))
    check_scores(dev, *branch_instance(seed, with_nan=False))


@pytest.mark.gpu
def test_score_special_nodes(dev):
    """f == inf (f_inv = 0), f_inv == inf next to x_hat = 0 (NaN) and next to x_hat = TINY (inf), f == 0, f1 == f2."""
    ref = check_scores(dev, *special_nodes_instance())
    assert np.isnan(ref).any() and np.isinf(ref).any()


@pytest.mark.gpu
def test_score_each_branch_pair_alone(dev):
    """Every branch pair on an arc of its own, between two nodes that carry an ordinary arc each (so the pair's node
    sums are not masked by anything else)."""
    pairs = branch_pairs()
    P = len(pairs)
    # arc p: 2p -> 2p+1 with the pair; arcs 2p+1 -> 2p+2 ... an ordinary path through all nodes
    tail = np.concatenate([2 * np.arange(P), np.arange(2 * P - 1)])
    head = np.concatenate([2 * np.arange(P) + 1, np.arange(1, 2 * P)])
    x = np.concatenate([[p[0] for p in pairs], np.full(2 * P - 1, 1.0)])
    u = np.concatenate([[p[1] for p in pairs], np.full(2 * P - 1, 5.0)])
    ref = check_scores(dev, tail.astype(np.int64), head.astype(np.int64), x, u, 2 * P)
    # u == inf gives NaN, as the get_sorted_flows docstring says
    assert np.isnan(ref[[q for q, p in enumerate(pairs) if p[1] == INF]]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [11, 12])
def test_score_hub_summation_order(dev, seed):
    """A hub of degree 2^17 + 5 and four nodes of degree ~1000 summed by the kernel in ascending arc id, as
    csr_matvec does: bit for bit (test_hub_sums_are_order_sensitive shows another order would change them)."""
    check_scores(dev, *hub_instance(seed))


def _sweep_cases():
    out = []
    for dn in (-1, 0, 1):
        for de in (-1, 0, 1):
            out.append(pytest.param(dn, de, id=f"nodes{dn:+d}-arcs{de:+d}"))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("dn,de", _sweep_cases())
def test_score_grid_stride_boundaries(dev, dn, de):
    """grid_for caps the grid at num_sms * 16 blocks: mcf_node_kernel covers num_sms * 16 * 128 nodes per sweep, the
    arc kernels num_sms * 16 * 256 arcs.  N and E at exactly one sweep and one off either way."""
    sms = num_sms()
    N = sms * 16 * 128 + dn
    E = sms * 16 * 256 + de
    tail, head, x, u = sweep_instance(N, E, 100 + 3 * dn + de)
    check_scores(dev, tail, head, x, u, N)


@pytest.mark.gpu
def test_score_through_the_manager_storage_forms(dev):
    """MCFManagerStd.get_sorted_flows with A as canonical CSR, as CSR with unsorted column indices, as CSC, and with
    stored zeros (no incidence: they touch no node sum even where x_hat is NaN): identical scores and queue, equal
    to the reference and to np.argsort(scores, kind="stable")[::-1] -- NaN scores sort last, so they lead the queue."""
    from smart_crossover.formats import MinCostFlow
    from smart_crossover.network_methods.net_manager import MCFManagerStd
    tail, head, x, u, N = branch_instance(5)
    E = tail.size
    A = incidence(tail, head, N)
    ref = mcf_scores_ref(x, u, A, tail, head)
    assert np.isnan(ref).any()
    rng = np.random.default_rng(5)
    # unsorted: every row's entries in a random order
    idx, dat = A.indices.copy(), A.data.copy()
    for v in range(N):
        lo, hi = A.indptr[v], A.indptr[v + 1]
        p = lo + rng.permutation(hi - lo)
        idx[lo:hi], dat[lo:hi] = idx[p], dat[p]
    A_uns = sp.csr_matrix((dat, idx, A.indptr.copy()), shape=A.shape)
    assert not A_uns.has_sorted_indices
    # stored zeros: at a node the arc does not touch, on NaN and on ordinary arcs
    nan_arcs = np.flatnonzero(np.isnan(xhat_ref(x, u)[0]))
    z_arc = np.concatenate([nan_arcs[:4], rng.choice(E, 8, replace=False)])
    z_row = np.array([next(r for r in range(N) if r not in (tail[k], head[k])) for k in z_arc])
    # built from (data, indices, indptr): a COO -> CSR conversion would sum and could drop the zeros
    coo = A.tocoo()
    rows = np.concatenate([coo.row, z_row])
    cols = np.concatenate([coo.col, z_arc])
    vals = np.concatenate([coo.data, np.zeros(z_arc.size)])
    o = np.lexsort((cols, rows))
    A_zero = sp.csr_matrix((vals[o], cols[o], np.searchsorted(rows[o], np.arange(N + 1))), shape=A.shape)
    assert A_zero.nnz == A.nnz + z_arc.size and (A_zero.data == 0).sum() == z_arc.size
    b = np.zeros(N)
    queue_ref = np.argsort(ref, kind="stable")[::-1]
    assert np.isnan(ref[queue_ref[0]])
    for form, M in (("csr", A), ("unsorted", A_uns), ("csc", A.tocsc()), ("stored_zeros", A_zero)):
        mgr = MCFManagerStd(MinCostFlow(M, b, np.ones(E), u))
        queue, scores = mgr.get_sorted_flows(x)
        same_bits(scores, ref)
        assert np.array_equal(queue, queue_ref), form


# ==== GPU: sx_price_arcs ===================================================================================
def pricer(dev, K, cap=None):
    import torch
    return dev.Pricer(torch.device("cuda"), K, cand_cap=cap, fused=False)


def one_pass(pr, calls):
    """reset, the given price_arcs calls (c, tail, head, vbasis, y, id0, rc_out), select, fetch."""
    pr.reset()
    for c, t, h, vb, y, id0, rc_out in calls:
        pr.price_arcs(c, t, h, vb, y, id0, TOL, rc_out)
    pr.select()
    res = pr.fetch()
    assert not pr.overflowed(res)
    return res


def check_summary(res, rc, K, id0=0):
    cnt, mn, ids, vals, nan = summary_ref(rc, K)
    assert res.n_violating == cnt
    assert np.float64(res.min_rc).tobytes() == np.float64(mn).tobytes()
    assert res.has_nan == nan and res.status == (NAN_RC if nan else 0)
    assert res.optimal == (cnt == 0 and not nan)
    if K:
        assert np.array_equal(res.topk_id, ids + id0)
        assert res.topk_rc.tobytes() == vals.tobytes()


def random_arcs(E, N, rng):
    tail = rng.integers(0, N, E).astype(np.int32)
    head = ((tail + 1 + rng.integers(0, N - 1, E)) % N).astype(np.int32)
    return tail, head


def layouts(c, tail, head, vb):
    """The same arc list under every dispatch: vector bulk + scalar tail (all aligned), then everything through the
    scalar kernel -- vbasis shifted by 1, 2 and 3 bytes, rc_out shifted by 8 bytes, all arrays shifted by one
    element -- and vbasis shifted by 4 bytes, which the vector kernel still takes.
    Yields (name, c_t, tail_t, head_t, vb_t, rc_out_t)."""
    import torch
    E = c.size
    ct, tt, ht = cu(c), cu(tail), cu(head)
    for name, vshift, rshift, all_shift in (("aligned", 0, 0, False), ("vbasis+1", 1, 0, False),
                                            ("vbasis+2", 2, 0, False), ("vbasis+3", 3, 0, False),
                                            ("vbasis+4", 4, 0, False), ("rc_out+8", 0, 1, False),
                                            ("all+1", 0, 0, True)):
        if all_shift:
            c2 = torch.empty(E + 1, dtype=torch.float64, device="cuda")[1:]
            t2 = torch.empty(E + 1, dtype=torch.int32, device="cuda")[1:]
            h2 = torch.empty(E + 1, dtype=torch.int32, device="cuda")[1:]
            c2.copy_(ct), t2.copy_(tt), h2.copy_(ht)
        else:
            c2, t2, h2 = ct, tt, ht
        v2 = None
        if vb is not None:
            v2 = torch.empty(E + 8, dtype=torch.int8, device="cuda")[vshift:vshift + E]
            v2.copy_(cu(vb))
        rc = torch.full((E + 2,), -7.0, dtype=torch.float64, device="cuda")[rshift:rshift + E]
        yield name, c2, t2, h2, v2, rc


def check_all_layouts(dev, c, tail, head, vb, y, K, id0=0):
    rc = rc_ref(c, tail, head, y, vb)
    yt = cu(y)
    pr = pricer(dev, K)
    for name, ct, tt, ht, vt, rct in layouts(c, tail, head, vb):
        res = one_pass(pr, [(ct, tt, ht, vt, yt, id0, rct)])
        same_bits(rct.cpu().numpy(), rc)
        check_summary(res, rc, K, id0)
    return rc


@pytest.mark.gpu
@pytest.mark.parametrize("E", [4099, 20003])
def test_price_non_finite_inputs(dev, E):
    """NaN in c, NaN at a tail dual and at a head dual, inf - inf in y[tail] - y[head], c = inf against that, -inf
    costs (violators at -inf): NaN is neither counted nor selected, sets SX_STATUS_NAN_RC and makes the pass not
    optimal, on every dispatch."""
    rng = np.random.default_rng(E)
    N = 500
    tail, head = random_arcs(E, N, rng)
    y = rng.random(N) * 10.0
    c = np.round(rng.random(E) * 12.0, 1)
    vb = rng.choice(np.array([-1, -2, 0], dtype=np.int8), E, p=[0.7, 0.2, 0.1])
    # node 1: NaN dual; nodes 2 (inf) and 3 (inf): arcs 2 -> 3 give inf - inf
    y[1], y[2], y[3] = NAN, INF, INF
    pick = rng.choice(E, 40, replace=False)
    c[pick[:5]] = NAN
    tail[pick[5:10]], head[pick[10:15]] = 1, 1
    tail[pick[15:25]], head[pick[15:25]] = 2, 3
    c[pick[20:25]] = INF                                                   # inf - NaN
    c[pick[25:30]] = -INF
    c[E - 2] = NAN                                                         # in the scalar tail too
    for K in (0, 64):
        rc = check_all_layouts(dev, c, tail, head, vb, y, K)
        assert np.isnan(rc).any() and np.isneginf(rc).any()


@pytest.mark.gpu
@pytest.mark.parametrize("E", [2048, 8195, 1_000_000])
def test_price_all_duals_nan(dev, E):
    """Duals that are all NaN (a failed solve): every rc is NaN, nothing is counted, the minimum is +inf (no
    reduced cost is a number) and the pass is not optimal."""
    rng = np.random.default_rng(E)
    N = 1000
    tail, head = random_arcs(E, N, rng)
    check_all_layouts(dev, rng.random(E), tail, head, None, np.full(N, NAN), 8)


@pytest.mark.gpu
def test_price_lone_nan_in_a_later_sweep(dev):
    """One NaN cost in the second grid sweep of each kernel, among arcs whose rc is all +1: by then every thread's
    running bound is 1 and lets no finite arc through, so only the unordered comparison sees the NaN."""
    import torch
    sms = num_sms()
    N = 1000
    for which, sweep in (("vector", sms * 3 * 2048), ("scalar", sms * 8 * 1024)):
        E = 2 * sweep
        rng = np.random.default_rng(E)
        tail, head = random_arcs(E, N, rng)
        c = np.full(E, 1.0)
        c[sweep + 777] = NAN
        rshift = 0 if which == "vector" else 1
        out = torch.empty(E + 1, dtype=torch.float64, device="cuda")[rshift:rshift + E]
        res = one_pass(pricer(dev, 16), [(cu(c), cu(tail), cu(head), None, cu(np.zeros(N)), 0, out)])
        rc = rc_ref(c, tail, head, np.zeros(N))
        same_bits(out.cpu().numpy(), rc)
        check_summary(res, rc, 16)
        assert res.has_nan and not res.optimal, which


@pytest.mark.gpu
def test_price_sign_of_zero(dev):
    """rc = +0.0 with vbasis == -2 must come out as -0.0 and -0.0 as +0.0, bitwise, on every dispatch; zeros are not
    violators and a zero minimum is reported as +0.0."""
    E, N = 4103, 64
    rng = np.random.default_rng(4)
    tail, head = random_arcs(E, N - 7, rng)
    tail, head = tail + 7, head + 7                                        # nodes 5 and 6 only where put below
    y = np.full(N, 1.5)
    y[5] = -0.0
    y[6] = 0.0
    c = np.zeros(E)
    c[rng.random(E) < 0.3] = -0.0
    tail[:20], head[:20] = 5, 6                                            # -0.0 - 0.0 = -0.0 in the dual difference
    vb = rng.choice(np.array([-1, -2, 0], dtype=np.int8), E)
    vb[-3:] = -2                                                           # negations in the scalar tail
    rc = check_all_layouts(dev, c, tail, head, vb, y, 16)
    assert np.all(rc == 0) and np.signbit(rc).any() and (~np.signbit(rc)).any()
    assert np.signbit(rc[vb == -2]).any() and np.signbit(rc[vb != -2]).any()


@pytest.mark.gpu
def test_price_tolerance_boundary(dev):
    """rc == -tol exactly is not a violator, nextafter(-tol, -inf) is; with and without the vbasis negation, in the
    vector bulk and in the scalar tail, and with everything through the scalar kernel."""
    E, N = 8195, 300
    rng = np.random.default_rng(8)
    tail, head = random_arcs(E, N, rng)
    y = np.zeros(N)
    c = rng.integers(1, 5, E).astype(np.float64)
    vb = np.full(E, -1, dtype=np.int8)
    below = np.nextafter(-TOL, -INF)
    above = np.nextafter(-TOL, INF)
    spots = np.concatenate([rng.choice(E - 4, 24, replace=False), [E - 3, E - 2, E - 1]])
    for q, k in enumerate(spots):
        kind = q % 6
        c[k] = (-TOL, TOL, below, -below, above, -above)[kind]
        vb[k] = -2 if kind % 2 else -1
    rc = check_all_layouts(dev, c, tail, head, vb, y, 64)
    assert (rc == -TOL).sum() >= 8 and (rc == below).sum() >= 8
    assert summary_ref(rc, 0)[0] == (rc == below).sum()


def _chunk_sizes():
    vec, sca = 256 * 8, 256 * 4
    out = []
    for base in (sca, vec, 2 * vec, 3 * vec, 5 * sca):
        out += [base + d for d in range(-3, 4)]
    return sorted(set(out))


@pytest.mark.gpu
def test_price_chunk_boundaries(dev):
    """E around the vector kernel's chunk (256 threads x 8 arcs), the scalar kernel's (256 x 4) and multiples of
    them, -3 .. +3, on every dispatch: rc bitwise and the summary.  The violators are spread to the last arc."""
    rng = np.random.default_rng(21)
    N = 700
    for E in _chunk_sizes():
        tail, head = random_arcs(E, N, rng)
        y = rng.random(N) * 4.0
        c = rng.integers(0, 5, E).astype(np.float64)
        vb = rng.choice(np.array([-1, -2, 0], dtype=np.int8), E, p=[0.6, 0.2, 0.2])
        check_all_layouts(dev, c, tail, head, vb, y, 32)


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["vector", "scalar"])
@pytest.mark.parametrize("d", [-1, 0, 1])
def test_price_grid_sweep_boundaries(dev, which, d):
    """One arc off either side of a whole grid sweep: num_sms * 3 blocks of 2048 arcs for the vector kernel,
    num_sms * 8 blocks of 1024 arcs for the scalar one (the list sent there with a shifted rc_out)."""
    import torch
    sms = num_sms()
    E = (sms * 3 * 2048 if which == "vector" else sms * 8 * 1024) + d
    rng = np.random.default_rng(E)
    N = 20000
    tail, head = random_arcs(E, N, rng)
    y = rng.random(N) * 10.0
    c = rng.random(E) * 12.0
    vb = rng.choice(np.array([-1, -2], dtype=np.int8), E, p=[0.9, 0.1])
    c[-1], vb[-1] = -50.0, -1                                              # the last arc is the most violating
    rc = rc_ref(c, tail, head, y, vb)
    rshift = 0 if which == "vector" else 1
    out = torch.empty(E + 1, dtype=torch.float64, device="cuda")[rshift:rshift + E]
    res = one_pass(pricer(dev, 64), [(cu(c), cu(tail), cu(head), cu(vb), cu(y), 0, out)])
    same_bits(out.cpu().numpy(), rc)
    check_summary(res, rc, 64)
    assert res.topk_id[0] == E - 1


def _split_list(E, rng):
    N = 3000
    tail, head = random_arcs(E, N, rng)
    y = rng.integers(0, 20, N).astype(np.float64)
    c = rng.integers(0, 25, E).astype(np.float64)
    vb = rng.choice(np.array([-1, -2, 0], dtype=np.int8), E, p=[0.7, 0.2, 0.1])
    c[-3:], vb[-3:] = -100.0, -1                                           # the scalar tail holds the top violators
    return c, tail, head, vb, y


@pytest.mark.gpu
@pytest.mark.parametrize("K", [0, 64, 1024, 3000])
def test_price_ids_past_2_31_and_accumulated_calls(dev, K):
    """One list priced with id0 = 3e9 reports ids past 2^31 (from both kernels); the same list split into three
    calls of one pass (consistent id0s, one aligned, two not) gives the single call's result, and both equal the
    reference."""
    import torch
    E = 50003
    rng = np.random.default_rng(K + 1)
    c, tail, head, vb, y = _split_list(E, rng)
    rc = rc_ref(c, tail, head, y, vb)
    ct, tt, ht, vt, yt = cu(c), cu(tail), cu(head), cu(vb), cu(y)
    pr = pricer(dev, K)
    out1 = torch.empty(E, dtype=torch.float64, device="cuda")
    single = one_pass(pr, [(ct, tt, ht, vt, yt, ID0_FAR, out1)])
    same_bits(out1.cpu().numpy(), rc)
    check_summary(single, rc, K, ID0_FAR)
    if K:
        assert single.topk_id.min() > 1 << 31 and (ID0_FAR + E - 1) in single.topk_id
    out3 = torch.full((E,), -1.0, dtype=torch.float64, device="cuda")
    cuts = [0, 4096, 4096 + 10001, E]
    calls = [(ct[a:b], tt[a:b], ht[a:b], vt[a:b], yt, ID0_FAR + a, out3[a:b]) for a, b in zip(cuts, cuts[1:])]
    split = one_pass(pr, calls)
    assert out3.cpu().numpy().tobytes() == out1.cpu().numpy().tobytes()
    assert split.n_violating == single.n_violating and split.status == single.status
    assert np.float64(split.min_rc).tobytes() == np.float64(single.min_rc).tobytes()
    assert np.array_equal(split.topk_id, single.topk_id) and split.topk_rc.tobytes() == single.topk_rc.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 1024, 3000])
def test_price_top_k_on_heavy_ties(dev, K):
    """Integer costs and duals: a few distinct reduced costs over 200 000 arcs, so the K-th value ties with
    thousands of arcs and the selection must finish on ascending ids.  K = 3000 > SX_TOPK_MAX_K takes the two-sort
    path.  Every dispatch."""
    E, N = 200_001, 4000
    rng = np.random.default_rng(K)
    tail, head = random_arcs(E, N, rng)
    y = rng.integers(0, 3, N).astype(np.float64)
    c = rng.integers(0, 4, E).astype(np.float64)
    vb = rng.choice(np.array([-1, -2], dtype=np.int8), E, p=[0.8, 0.2])
    rc = check_all_layouts(dev, c, tail, head, vb, y, K)
    cnt, mn, ids, vals, _ = summary_ref(rc, K)
    assert cnt > 10 * K and (rc == vals[-1]).sum() > K


@pytest.mark.gpu
def test_price_candidate_overflow_repeat(dev):
    """A pricer whose candidate buffer (512) holds fewer than the violators tied at the K-th value: the pass
    overflows, the buffer grows and the pass is repeated until the answer is complete."""
    import torch
    E, N, K = 100_003, 2000, 100
    rng = np.random.default_rng(3)
    tail, head = random_arcs(E, N, rng)
    y = np.zeros(N)
    c = np.where(rng.random(E) < 0.5, -1.0, 1.0)
    pr = pricer(dev, K, cap=512)
    res = dev.price_arcs(cu(c), cu(tail), cu(head), cu(y), K=K, want_rc=True, pricer=pr)
    rc = rc_ref(c, tail, head, y)
    same_bits(res.rc.cpu().numpy(), rc)
    check_summary(res, rc, K)
    assert pr.cap > 512
    cap = pr.cap
    res = dev.price_arcs(cu(c), cu(tail), cu(head), cu(y), K=K, pricer=pr)       # fits now: no further growth
    check_summary(res, rc, K)
    assert pr.cap == cap


@pytest.mark.gpu
@pytest.mark.parametrize("K", [0, 50, 3000])
def test_price_manager_after_bigm(dev, K):
    """MCFManagerStd.price and get_reduced_cost_for_original_mcf after extend_by_bigM against `c - A.T @ y` (negated
    at the arcs fixed at their upper bound) on the explicitly extended A: the artificial arcs' endpoints, which the
    manager takes from the host instead of scanning A, must be the ones A has."""
    from smart_crossover.formats import MinCostFlow
    from smart_crossover.network_methods.net_manager import MCFManagerStd
    N, E = 400, 5000
    tail, head, b, c, u = cases.netgen_like(N, E, 77)
    rng = np.random.default_rng(77)
    mgr = MCFManagerStd(MinCostFlow(incidence(tail, head, N), b, c, u))
    ids = rng.permutation(E)
    mgr.fix_variables(np.sort(ids[:1000]), np.sort(ids[1000:1600]))
    mgr.extend_by_bigM(1e6)
    mgr.set_initial_basis()
    A_ext = sp.csr_matrix(mgr.mcf.A)
    assert A_ext.shape == (N + 1, E + N)
    vb = np.asarray(mgr.basis.vbasis)
    assert (vb == -2).sum() == 600
    for scale in (1.0, 1e4):
        y = np.round(rng.normal(0, scale, N + 1), 2)
        with np.errstate(invalid="ignore"):
            rc = mgr.mcf.c - A_ext.T @ y
        rc[vb == -2] = -rc[vb == -2]
        res = mgr.price(y, K=K, want_rc=True)
        same_bits(res.rc.cpu().numpy(), rc)
        check_summary(res, rc, K)
        same_bits(mgr.get_reduced_cost_for_original_mcf(y), rc)

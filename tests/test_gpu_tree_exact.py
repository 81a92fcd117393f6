"""The tree-basis kernels against exact references.

sx_kruskal picks the tree arcs, sx_tree_potentials gives the duals of the tree basis and sx_tree_flows its
primal flows.  Every check here compares with an exact host computation, never with another fp64 code:

  * Kruskal: the forest of the sequential oracle over the same `korder` (arc ids ascending, bit-exact), at an
    N in every launch variant of sx_kruskal (one CTA with the survivor lists in shared memory, one CTA with
    them in global memory, cooperative at 1 CTA/SM, cooperative at up to 4 CTAs/SM), on adversarial orders
    (paths along / against / across the order, stars, self-loops and parallel arcs, forests, completion at
    and just after a chunk boundary, OT prefixes) and under every first-chunk schedule.
  * Potentials: BFS from the root in exact integer arithmetic on a common binary grid.  On costs of a
    common dyadic grid every partial sum the kernel forms is exact, so it must be bit-exact there; on real
    costs its error is bounded normwise, 2 ceil(log2 H) eps max|y| (POT_ULPS_PER_ROUND below).
  * Flows: exact subtree sums.  The flow of an arc is within 1 ulp of the exact sum wherever
    sum|b| / |sum| <= 2^50 / H (H = 2 (N - 1) tour positions), and within 1/2 ulp + 2^-103 H sum|b| everywhere;
    exact zeros come out as +-0.0.

The tests without the `gpu` marker check the references themselves and show, on a host emulation of the
kernels' exact association, that a plain-double prefix sum in place of the double-double one fails the
flow bound.
"""
import math

import numpy as np
import pytest
import scipy.sparse as sp
from scipy.sparse import csgraph

from oracle import network_oracle as orc

EPS = 2.0 ** -52
TOUR_SMALL_H = 4096          # kTourSmallH in sx_tree.cu: one CTA ranks tours of up to this many half-edges
# Normwise error bound of the potentials on real costs, in units of eps * max|y_exact| per pointer-jumping
# round (ceil(log2 H) rounds).  Measured on a B200 (1000 W limit) over test_potentials_real_costs_normwise:
# at most 0.25 per round up to N = 1e5 and 0.86 per round (17.2 eps * max|y|) at N = 4e5.
POT_ULPS_PER_ROUND = 2


# ==== exact references ==================================================================================
def to_grid(x, headroom=0):
    """Doubles -> (integers m, E) with x = m * 2^-E exactly: int64 when they fit with `headroom` bits to
    spare for sums, else Python ints."""
    x = np.asarray(x, dtype=np.float64)
    nz = x[x != 0]
    if nz.size == 0:
        return np.zeros(x.size, dtype=np.int64), 0
    mant, ex = np.frexp(nz)                               # nz = mant * 2^ex, 0.5 <= |mant| < 1
    m53 = (mant * 2.0 ** 53).astype(np.int64)             # exact
    # strip trailing zero bits so that E is as small as the data allows
    tz = np.zeros(nz.size, dtype=np.int64)
    t = np.abs(m53)
    for _ in range(53):
        odd = (t & 1) == 1
        if odd.all():
            break
        t = np.where(odd, t, t >> 1)
        tz += ~odd
    odd_m = m53 >> tz                                     # nz = odd_m * 2^(ex - 53 + tz)
    E = max(0, int((53 - ex - tz).max()))
    shift = (ex - 53 + tz + E).astype(np.int64)           # >= 0
    bits = 53 - tz + shift
    if bits.max() + headroom < 62:
        out = np.zeros(x.size, dtype=np.int64)
        out_nz = odd_m << shift
    else:
        out = np.zeros(x.size, dtype=object)
        out_nz = np.array([int(m) << int(s) for m, s in zip(odd_m, shift)], dtype=object)
    out[x != 0] = out_nz
    return out, E


def grid_to_float(m, E):
    """Correctly rounded m * 2^-E (Python's int / int division rounds correctly)."""
    d = 1 << E
    return np.array([int(v) / d for v in m], dtype=np.float64)


def tree_bfs(plus, minus, N, root):
    """BFS of the tree (plus[t], minus[t]) from `root`: (order, child node of every arc, True where the
    child is the arc's plus end).  ValueError if the arcs are not a spanning tree of the N nodes."""
    plus = np.asarray(plus, dtype=np.int64)
    minus = np.asarray(minus, dtype=np.int64)
    T = plus.size
    if T != N - 1:
        raise ValueError("not a spanning tree: %d arcs on %d nodes" % (T, N))
    if N == 1:
        return np.zeros(1, dtype=np.int64), np.zeros(0, dtype=np.int64), np.zeros(0, dtype=bool)
    g = sp.coo_matrix((np.ones(T), (plus, minus)), shape=(N, N)).tocsr()
    order, pred = csgraph.breadth_first_order(g, root, directed=False, return_predecessors=True)
    if order.size != N:
        raise ValueError("not a spanning tree: disconnected")
    plus_child = pred[plus] == minus
    child = np.where(plus_child, plus, minus)
    if not (plus_child | (pred[minus] == plus)).all() or np.bincount(child, minlength=N).max() > 1 \
            or (child == root).any():
        raise ValueError("not a spanning tree: cycle")
    return order, child, plus_child


def exact_potentials(plus, minus, cost, N, root):
    """y with y[root] = 0 and y[plus] - y[minus] = cost on every arc, exactly: (m, E) with y = m * 2^-E.
    Integer pointer jumping over the parents (ceil(log2 N) rounds), so large trees stay fast."""
    order, child, plus_child = tree_bfs(plus, minus, N, root)
    c, E = to_grid(cost, headroom=math.ceil(math.log2(max(N, 2))) + 1)
    par = np.arange(N, dtype=np.int64)
    par[child] = np.where(plus_child, minus, plus)
    val = np.zeros(N, dtype=c.dtype)
    val[child] = np.where(plus_child, c, -c)
    for _ in range(max(1, math.ceil(math.log2(max(N, 2))))):
        val = val + val[par]
        par = par[par]
    return val, E


def exact_subtree_flows(plus, minus, b, N, root):
    """x with B x = b on every node but the root (B: +1 at plus, -1 at minus): the flow of an arc is the
    exact sum of b over the subtree below it, + when the subtree hangs at its plus end.  (m, E) with
    x = m * 2^-E, Python ints."""
    order, child, plus_child = tree_bfs(plus, minus, N, root)
    bm, E = to_grid(b)
    par = np.arange(N, dtype=np.int64)
    par[child] = np.where(plus_child, minus, plus)
    sub = [int(v) for v in bm]
    parl = par.tolist()
    for v in order[:0:-1].tolist():                       # reverse BFS order: children before parents
        sub[parl[v]] += sub[v]
    flows = [sub[ch] if pc else -sub[ch] for ch, pc in zip(child.tolist(), plus_child.tolist())]
    return flows, E


def ulp_errors(got, m, E):
    """For doubles `got` and exact values m * 2^-E: (|got - exact| in units of 2^-E as ints, the exact
    values rounded, ulp of the rounded exact values)."""
    exact = grid_to_float(m, E)
    err = []
    for g, v in zip(got.tolist(), m):
        p, q = float(g).as_integer_ratio()               # q is a power of two
        if (1 << E) % q:
            err.append(None)                              # finer than the grid: cannot be a rounded grid sum
        else:
            err.append(abs(p * ((1 << E) // q) - int(v)))
    return err, exact, np.array([math.ulp(v) for v in exact])


def within(err, bound, E):
    """err (ints, units of 2^-E) <= bound (doubles), exactly."""
    out = []
    for e, bd in zip(err, bound.tolist()):
        if e is None:
            out.append(False)
            continue
        p, q = float(bd).as_integer_ratio()
        out.append(e * q <= p * (1 << E))
    return np.array(out, dtype=bool)


# ==== tree generators ====================================================================================
SHAPES = ["path", "path_reversed", "path_shuffled", "star", "caterpillar", "broom", "binary", "recursive"]


def tree_shape(shape, N, rng):
    """Undirected edges (u, v) of a tree on nodes 0..N-1, in the order they are listed."""
    i = np.arange(1, N, dtype=np.int64)
    if shape == "path":                          # labels and arcs in order along the path
        u, v = i - 1, i
    elif shape == "path_reversed":               # arcs listed from the far end, each pointing backwards
        u, v = i[::-1], i[::-1] - 1
    elif shape == "path_shuffled":               # a path through random labels, arcs in random order
        p = rng.permutation(N)
        u, v = p[i - 1], p[i]
    elif shape == "star":                        # one node of degree N-1, away from both ends of the labels
        hub = N // 2
        leaves = np.delete(np.arange(N), hub)
        u, v = np.full(N - 1, hub), leaves
    elif shape == "caterpillar":                 # a spine with one leg on every spine node
        m = (N + 1) // 2
        u = np.concatenate([np.arange(m - 1), np.arange(N - m)])
        v = np.concatenate([np.arange(1, m), np.arange(m, N)])
    elif shape == "broom":                       # a handle path ending in a star
        m = max(N // 2, 1)
        u = np.concatenate([np.arange(m - 1), np.full(N - m, m - 1)])
        v = np.concatenate([np.arange(1, m), np.arange(m, N)])
    elif shape == "binary":                      # complete binary tree in heap order
        u, v = (i - 1) // 2, i
    elif shape == "recursive":                   # random recursive tree, random labels
        par = (rng.random(N - 1) * i).astype(np.int64)
        p = rng.permutation(N)
        u, v = p[par], p[i]
    else:
        raise ValueError(shape)
    u, v = np.asarray(u, dtype=np.int64), np.asarray(v, dtype=np.int64)
    if shape not in ("path", "path_reversed"):
        o = rng.permutation(N - 1)
        u, v = u[o], v[o]
    return u, v


def pick_root(kind, plus, minus, N, rng):
    deg = np.bincount(np.concatenate([plus, minus]), minlength=N)
    if kind == "last":
        return N - 1
    if kind == "first":
        return 0
    if kind == "hub":
        return int(np.argmax(deg))
    if kind == "leaf":
        return int(rng.choice(np.flatnonzero(deg == 1)))
    raise ValueError(kind)


ROOTS = ["last", "first", "hub", "leaf"]


def orient(u, v, rng):
    """Random orientation: (plus, minus)."""
    flip = rng.random(u.size) < 0.5
    return np.where(flip, v, u), np.where(flip, u, v)


def arc_list(plus, minus, plus_is_tail, rng, extra=None):
    """The tree as a subset of a larger arc list: (tail, head, tree ids), with `extra` other arcs (valid ids,
    random positions) that the kernels must not touch."""
    T = plus.size
    extra = T // 3 + 1 if extra is None else extra
    E = T + extra
    N = int(max(plus.max(initial=0), minus.max(initial=0))) + 1
    ids = rng.permutation(E)[:T]
    tail = rng.integers(0, N, E).astype(np.int64)
    head = rng.integers(0, N, E).astype(np.int64)
    tail[ids] = plus if plus_is_tail else minus
    head[ids] = minus if plus_is_tail else plus
    return tail, head, ids.astype(np.int64)


def ot_tree(S, D, rng):
    """Maximum-weight spanning tree of random weights on the complete bipartite OT graph: arc ids k with
    plus = S + k % D, minus = k / D."""
    tree = orc.max_weight_spanning_tree(rng.random(S * D), S, D, drop_zero_weight=False)
    assert tree.size == S + D - 1
    return tree, S + tree % D, tree // D


# ==== host emulation of the kernels' association (sx_tree.cu) ============================================
def emulate_tour(plus, minus, N, root):
    """The Euler tour of tree_tour_kernel: half-edge 2t goes minus -> plus, 2t+1 plus -> minus; the
    successor of u -> v is the half-edge after v -> u in v's adjacency (half-edges sorted stably by
    origin), the tour is cut at the root's first half-edge.  Returns (rank, 1-based, 0 where unreached;
    dest) of every half-edge, like the kernel's ranking with the unreached ones marked."""
    T = plus.size
    H = 2 * T
    origin = np.empty(H, dtype=np.int64)
    dest = np.empty(H, dtype=np.int64)
    origin[0::2], dest[0::2] = minus, plus
    origin[1::2], dest[1::2] = plus, minus
    ho = np.argsort(origin, kind="stable")
    so = origin[ho]
    pos = np.empty(H, dtype=np.int64)
    pos[ho] = np.arange(H)
    first = np.full(N, -1, dtype=np.int64)
    starts = np.flatnonzero(np.r_[True, so[1:] != so[:-1]])
    first[so[starts]] = starts
    p2 = pos[np.arange(H) ^ 1] + 1
    wrap = (p2 >= H)
    p2c = np.minimum(p2, H - 1)
    wrap |= so[p2c] != dest
    p2 = np.where(wrap, first[dest], p2)
    succ = ho[p2]
    rank = np.zeros(H, dtype=np.int64)
    if first[root] < 0:
        return rank, dest
    h = int(ho[first[root]])
    succl = succ.tolist()
    r = 1
    while rank[h] == 0:
        rank[h] = r
        r += 1
        h = succl[h]
    return rank, dest


def _dd_add(hi, lo, b):
    s = hi + b
    bb = s - hi
    e = (hi - (s - bb)) + (b - bb)
    lo2 = lo + e
    hi2 = s + lo2
    return hi2, lo2 - (hi2 - s)


def emulate_flows(plus, minus, b, N, root, double_double=True):
    """sx_tree_flows on the host with the kernels' exact association: scatter into tour positions, the
    1024-thread chunked scan of flow_scan_kernel, prefix differences of flow_finalize_kernel.  With
    double_double=False the prefix sums are plain doubles (what the kernel would compute without dd_add)."""
    rank, dest = emulate_tour(plus, minus, N, root)
    T = plus.size
    H = 2 * T
    assert (rank > 0).all()
    ra, rb = rank[0::2], rank[1::2]
    a_down = ra < rb
    r_down = np.where(a_down, ra, rb) - 1
    r_up = np.where(a_down, rb, ra) - 1
    w = np.zeros(H)
    w[r_down] = b[np.where(a_down, dest[0::2], dest[1::2])]
    chunk = (H + 1023) // 1024
    lo_i = np.arange(1024) * chunk
    hi_i = np.minimum(lo_i + chunk, H)
    acc_hi, acc_lo = np.zeros(1024), np.zeros(1024)
    for k in range(chunk):
        m = lo_i + k < hi_i
        x = np.where(m, w[np.minimum(lo_i + k, H - 1)], 0.0)
        if double_double:
            nh, nl = _dd_add(acc_hi, acc_lo, x)
        else:
            nh, nl = acc_hi + x, acc_lo
        acc_hi, acc_lo = np.where(m, nh, acc_hi), np.where(m, nl, acc_lo)
    ex_hi, ex_lo = np.zeros(1024), np.zeros(1024)
    run_hi, run_lo = 0.0, 0.0
    for t in range(1024):
        ex_hi[t], ex_lo[t] = run_hi, run_lo
        if double_double:
            run_hi, run_lo = _dd_add(*_dd_add(run_hi, run_lo, acc_hi[t]), acc_lo[t])
        else:
            run_hi = run_hi + acc_hi[t]
    phi, plo = np.zeros(H), np.zeros(H)
    acc_hi, acc_lo = ex_hi, ex_lo
    for k in range(chunk):
        m = lo_i + k < hi_i
        idx = np.minimum(lo_i + k, H - 1)
        if double_double:
            acc_hi, acc_lo = _dd_add(acc_hi, acc_lo, np.where(m, w[idx], 0.0))
        else:
            acc_hi = acc_hi + np.where(m, w[idx], 0.0)
        phi[idx[m]], plo[idx[m]] = acc_hi[m], acc_lo[m]
    top_hi, top_lo = phi[r_up], plo[r_up]
    has = r_down > 0
    prev = np.maximum(r_down - 1, 0)
    if double_double:
        h2, l2 = _dd_add(*_dd_add(top_hi, top_lo, -phi[prev]), -plo[prev])
    else:
        h2, l2 = top_hi - phi[prev], top_lo
    top_hi, top_lo = np.where(has, h2, top_hi), np.where(has, l2, top_lo)
    sub = top_hi + top_lo
    return np.where(a_down, sub, -sub)


def emulate_potentials(plus, minus, cost, N, root):
    """sx_tree_potentials on the host: Wyllie pointer jumping over the tour, ceil(log2 H) synchronous rounds."""
    rank, dest = emulate_tour(plus, minus, N, root)
    H = 2 * plus.size
    wgt = np.empty(H)
    wgt[0::2], wgt[1::2] = cost, -cost
    order = np.argsort(rank)
    pred = np.full(H, -1, dtype=np.int64)
    pred[order[1:]] = order[:-1]
    s = wgt.copy()
    rounds = max(1, math.ceil(math.log2(H)))
    for _ in range(rounds):
        has = pred >= 0
        pp = np.maximum(pred, 0)
        s = np.where(has, s[pp] + s, s)
        pred = np.where(has, pred[pp], pred)
    y = np.zeros(N)
    ra, rb = rank[0::2], rank[1::2]
    down = np.where(ra < rb, 2 * np.arange(plus.size), 2 * np.arange(plus.size) + 1)
    y[dest[down]] = s[down]
    y[root] = 0.0
    return y


# ==== data ===============================================================================================
def dyadic_costs(n, rng, span=24):
    """Costs k * 2^-20 with |k| < 2^span: every partial sum of a tour of up to 2^(53-span-1) half-edges
    is exact in fp64."""
    return rng.integers(-(1 << span) + 1, 1 << span, n).astype(np.float64) * 2.0 ** -20


def mixed_costs(n, rng):
    """Mostly O(1) costs with 1% of them scaled by 1e6 (a few expensive arcs)."""
    c = rng.random(n) + 0.01
    c[rng.random(n) < 0.01] *= 1e6
    return c


def wide_supplies(N, rng, decades=12):
    """Supplies of random sign and magnitudes spread over `decades` decades (1e-6 .. 1e6)."""
    mag = 10.0 ** rng.uniform(-decades / 2, decades / 2, N)
    return np.where(rng.random(N) < 0.5, -mag, mag) * (1.0 + rng.random(N))


def flow_bounds(m, E, got, H, abs_b_sum):
    """(ok within 1 ulp where the 2^50/H rule applies, ok against the general bound, mask of the rule)."""
    err, exact, ulp = ulp_errors(got, m, E)
    ratio = np.divide(abs_b_sum, np.abs(exact), out=np.full(exact.size, np.inf), where=exact != 0)
    rule = ratio <= 2.0 ** 50 / H
    one_ulp = within(err, ulp, E)
    general = within(err, 0.5 * ulp + 2.0 ** -103 * H * abs_b_sum, E)
    return one_ulp, general, rule, exact


# ==== CPU: the references themselves ====================================================================
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("N", [2, 3, 17, 300])
def test_exact_potentials_match_oracle_on_integer_costs(shape, N):
    """Integer costs: the sequential fp64 oracle is exact, so it must equal the exact reference; and the
    reference satisfies y[plus] - y[minus] = cost exactly, y[root] = 0."""
    rng = np.random.default_rng(N * 31 + len(shape))
    plus, minus = orient(*tree_shape(shape, N, rng), rng)
    cost = rng.integers(-1000, 1000, N - 1).astype(np.float64)
    for kind in ROOTS:
        root = pick_root(kind, plus, minus, N, rng)
        m, E = exact_potentials(plus, minus, cost, N, root)
        y = grid_to_float(m, E)
        assert np.array_equal(y, orc.tree_potentials(plus, minus, cost, N, root))
        c, Ec = to_grid(cost)
        assert Ec == E and m[root] == 0
        assert all(int(m[p]) - int(m[q]) == int(cc) for p, q, cc in zip(plus, minus, c))


def test_exact_potentials_fractional_costs_satisfy_the_arc_equations():
    rng = np.random.default_rng(5)
    N = 2000
    plus, minus = orient(*tree_shape("recursive", N, rng), rng)
    cost = mixed_costs(N - 1, rng)
    root = pick_root("leaf", plus, minus, N, rng)
    m, E = exact_potentials(plus, minus, cost, N, root)
    c, Ec = to_grid(cost)
    assert E == Ec and m[root] == 0
    assert all(int(m[p]) - int(m[q]) == int(cc) for p, q, cc in zip(plus, minus, c))
    # the fp64 oracle is close to it normwise
    y = grid_to_float(m, E)
    assert np.abs(orc.tree_potentials(plus, minus, cost, N, root) - y).max() <= 1e-12 * np.abs(y).max()


@pytest.mark.parametrize("S,D", [(1, 1), (2, 3), (30, 51), (200, 150)])
def test_exact_flows_match_oracle_on_integer_supplies(S, D):
    """OT trees, integer supplies, root N-1: the oracle's leaf elimination is exact, so it equals the
    exact subtree sums; and B x = b holds exactly on every node but the root."""
    rng = np.random.default_rng(S * 7 + D)
    tree, plus, minus = ot_tree(S, D, rng)
    s = rng.integers(1, 1000, S).astype(np.float64)
    d = rng.integers(1, 1000, D).astype(np.float64)
    d[-1] += s.sum() - d.sum()
    b = np.concatenate([-s, d])
    m, E = exact_subtree_flows(plus, minus, b, S + D, S + D - 1)
    assert E == 0
    assert np.array_equal(np.array(m, dtype=np.float64), orc.ot_tree_flows(tree, s, d))
    _check_conservation(plus, minus, m, b, S + D, S + D - 1)


def _check_conservation(plus, minus, m, b, N, root):
    """B x = b exactly on every node but the root (x = m * 2^-E on the grid of b)."""
    bm, _ = to_grid(b)
    bal = [0] * N
    for p, q, x in zip(plus.tolist(), minus.tolist(), m):
        bal[p] += x
        bal[q] -= x
    assert all(bal[v] == int(bm[v]) for v in range(N) if v != root)


@pytest.mark.parametrize("shape", ["path_shuffled", "star", "broom", "recursive"])
def test_exact_flows_conservation_any_root_unbalanced(shape):
    """Wide-span real supplies, Sum b != 0, every root kind: B x = b holds exactly off the root."""
    rng = np.random.default_rng(11)
    N = 700
    plus, minus = orient(*tree_shape(shape, N, rng), rng)
    b = wide_supplies(N, rng)
    for kind in ROOTS:
        root = pick_root(kind, plus, minus, N, rng)
        m, E = exact_subtree_flows(plus, minus, b, N, root)
        _check_conservation(plus, minus, m, b, N, root)


def test_tree_bfs_rejects_non_trees():
    with pytest.raises(ValueError):
        tree_bfs(np.array([0, 1]), np.array([1, 0]), 3, 0)          # parallel arcs, node 2 isolated
    with pytest.raises(ValueError):
        tree_bfs(np.array([0, 1, 2]), np.array([1, 2, 0]), 4, 0)     # triangle + isolated node
    with pytest.raises(ValueError):
        tree_bfs(np.array([0]), np.array([1]), 3, 0)                 # too few arcs


def test_plain_double_scan_fails_the_flow_bound():
    """On the host emulation of the kernels' association, the double-double scan meets the flow bound that
    test_tree_flows_wide_supplies asserts, and the same scan in plain doubles does not: that test tells
    the two apart."""
    rng = np.random.default_rng(2050)
    for shape, N in (("recursive", 2050), ("path_shuffled", 5000)):
        plus, minus = orient(*tree_shape(shape, N, rng), rng)
        b = wide_supplies(N, rng)
        root = pick_root("leaf", plus, minus, N, rng)
        m, E = exact_subtree_flows(plus, minus, b, N, root)
        H = 2 * (N - 1)
        abs_b = float(np.abs(np.delete(b, root)).sum())
        dd = emulate_flows(plus, minus, b, N, root, double_double=True)
        one, gen, rule, _ = flow_bounds(m, E, dd, H, abs_b)
        assert rule.sum() > N // 4
        assert one[rule].all() and gen.all()
        plain = emulate_flows(plus, minus, b, N, root, double_double=False)
        one, gen, rule, _ = flow_bounds(m, E, plain, H, abs_b)
        assert (~one[rule]).sum() > 10


def test_emulated_tour_of_a_non_spanning_single_face():
    """Three parallel arcs between nodes 0 and 1 with a path hanging off node 1, and two isolated nodes:
    N - 1 arcs, and the successor rule puts all of the half-edges into the root's tour.  Every half-edge is
    ranked, so only the isolated nodes (no half-edge at all) reveal that this is not a spanning tree."""
    plus, minus, N = non_spanning_single_face(40)
    rank, _ = emulate_tour(plus, minus, N, 0)
    assert (rank > 0).all() and sorted(rank.tolist()) == list(range(1, 2 * plus.size + 1))


def non_spanning_single_face(N):
    """N - 1 arcs on N nodes: 3 parallel arcs 0-1, a path 1 - 2 - ... - (N-3), nodes N-2 and N-1 isolated."""
    k = np.arange(2, N - 2)
    plus = np.concatenate([[1, 0, 1], k])
    minus = np.concatenate([[0, 1, 0], k - 1])
    return plus.astype(np.int64), minus.astype(np.int64), N


def non_spanning_cases(N):
    """Non-spanning inputs of N - 1 arcs on N nodes with valid ids: (name, plus, minus, root)."""
    k = np.arange(N - 1)
    cyc_p, cyc_m = k, (k + 1) % (N - 1)                     # cycle on 0..N-2, node N-1 isolated
    out = [("cycle+isolated", cyc_p, cyc_m, 0), ("isolated-root", cyc_p, cyc_m, N - 1)]
    # triangle 0-1-2 and a path over 3..N-1: every node has an arc, the path's half-edges are never reached
    tri_p, tri_m = np.array([0, 1, 2]), np.array([1, 2, 0])
    pth = np.arange(3, N - 1)
    out.append(("triangle+path", np.concatenate([tri_p, pth]), np.concatenate([tri_m, pth + 1]), 1))
    if N >= 6:
        sp_, sm_, _ = non_spanning_single_face(N)
        out.append(("single-face", sp_, sm_, 0))
    return out


def test_non_spanning_cases_are_not_trees():
    for N in (6, 2049, 2050):
        for name, p, m, root in non_spanning_cases(N):
            assert p.size == N - 1 and p.max() < N and m.max() < N and p.min() >= 0, name
            with pytest.raises(ValueError):
                tree_bfs(p, m, N, root)


# ==== GPU fixtures =======================================================================================
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


def cu_korder(korder):
    import torch
    return torch.from_numpy(np.ascontiguousarray(korder, dtype=np.int64).astype(np.uint32).view(np.int32)).cuda()


@pytest.fixture
def kr_tuning(dev):
    """Sets the process-wide first-chunk schedule of sx_kruskal; always restores the default."""
    from smart_crossover._native import lib

    def set_q(q):
        assert lib.sx_kruskal_set_tuning(q) == 0
    try:
        yield set_q
    finally:
        assert lib.sx_kruskal_set_tuning(0) == 0


def tour_path(N):
    return "smem" if 2 * (N - 1) <= TOUR_SMALL_H else "coop"


# ==== Kruskal =============================================================================================
KR_QS = [0, 1, 4, 64]


def kr_variant(N):
    """Which launch of sx_kruskal runs at N (sx_kruskal.cu)."""
    if N <= 16000:
        forest = ((N * 12 + 15) & ~15) + 16
        lists = (200 * 1024 - forest) // 24 if forest < 200 * 1024 else 0
        return "cta-smemlists" if lists >= 4096 else "cta-globallists"
    return "coop1" if N <= (1 << 18) else "coop4"


def kr_chunk_ends(N, q, upto):
    """Ends of the chunks of `korder` that sx_kruskal visits at N under first-chunk schedule q."""
    qe = q if q > 0 else (2 if N >= (1 << 18) else (8 if N >= (1 << 14) else 16))
    first = max(1024, (N * qe + 3) // 4)
    cap = max(8 * N, 1 << 22)
    if N <= 16000:
        forest = ((N * 12 + 15) & ~15) + 16
        lists = (200 * 1024 - forest) // 24 if forest < 200 * 1024 else 0
        if lists >= 4096:
            cap = min(cap, lists)
    ends, pos, cs = [], 0, min(first, cap)
    while pos < upto:
        pos += cs
        ends.append(pos)
        cs = min(2 * cs, cap)
    return ends


def random_tree_arcs(N, rng):
    u, v = tree_shape("recursive", N, rng)
    return orient(u, v, rng)


def kr_family(family, N, rng, q=0):
    """(tail, head, korder) of an arc-list graph on N nodes."""
    idx = np.arange(N - 1, dtype=np.int64)
    if family in ("path_along", "path_against"):
        tail, head = idx, idx + 1
        korder = idx if family == "path_along" else idx[::-1].copy()
    elif family == "path_random":
        p = rng.permutation(N)
        o = rng.permutation(N - 1)
        tail, head = p[idx][o], p[idx + 1][o]
        korder = rng.permutation(N - 1)
    elif family in ("star_hub0", "star_hubN"):
        hub = 0 if family == "star_hub0" else N - 1
        leaves = np.delete(np.arange(N), hub)
        tail, head = orient(np.full(N - 1, hub), leaves, rng)
        korder = rng.permutation(N - 1)
    elif family == "loops_parallel":
        tp, tm = random_tree_arcs(N, rng)
        loops = rng.integers(0, N, N // 2 + 1)
        dup = rng.integers(0, N - 1, N // 2 + 1)
        tail = np.concatenate([tp, loops, tm[dup]])          # parallel copies point the other way
        head = np.concatenate([tm, loops, tp[dup]])
        korder = rng.permutation(tail.size)
    elif family == "forest":
        k = max(2, N // 100)                                 # components
        tp, tm = random_tree_arcs(N, rng)
        keep = np.sort(rng.permutation(N - 1)[:N - k])
        tp, tm = tp[keep], tm[keep]
        # redundant arcs inside the components: parallel copies and self-loops
        dup = rng.integers(0, max(tp.size, 1), N // 3 + 1) if tp.size else np.zeros(0, dtype=np.int64)
        loops = rng.integers(0, N, N // 3 + 1)
        tail = np.concatenate([tp, tp[dup], loops])
        head = np.concatenate([tm, tm[dup], loops])
        korder = rng.permutation(tail.size)
    elif family in ("complete_at_chunk_end", "complete_after_chunk_end"):
        # the forest gets its last arc as the last arc of a chunk, or as the first arc of the next one;
        # every other position before it holds an arc that closes a cycle, and more arcs follow it
        ends = kr_chunk_ends(N, q, N - 1)
        P = ends[-1] - 1 if family == "complete_at_chunk_end" else ends[-1]
        tp, tm = random_tree_arcs(N, rng)
        last = rng.integers(0, N - 1)
        others = np.delete(np.arange(N - 1), last)
        slots = np.sort(rng.permutation(P)[:N - 2])          # positions of the other tree arcs
        is_tree = np.zeros(P, dtype=bool)
        is_tree[slots] = True
        seq = np.empty(P, dtype=np.int64)
        seq[slots] = rng.permutation(others)
        n_red = P - (N - 2)
        trail = N // 2 + 1
        # redundant arcs: a reversed copy of a tree arc placed before it, else a self-loop
        placed = seq[slots]
        placed_before = np.cumsum(is_tree)[~is_tree]
        red_src = np.full(n_red, -1, dtype=np.int64)
        if placed.size:
            pick = np.minimum((rng.random(n_red) * placed_before).astype(np.int64), placed.size - 1)
            red_src = np.where(placed_before > 0, placed[pick], -1)
        loops = rng.integers(0, N, n_red + trail)
        tail = np.concatenate([tp, np.where(red_src >= 0, tm[np.maximum(red_src, 0)], loops[:n_red]),
                               loops[n_red:]])
        head = np.concatenate([tm, np.where(red_src >= 0, tp[np.maximum(red_src, 0)], loops[:n_red]),
                               loops[n_red:]])
        seq[~is_tree] = N - 1 + np.arange(n_red)
        trailing = N - 1 + n_red + rng.permutation(trail)
        korder = np.concatenate([seq, [last], trailing])
        # trailing arcs include copies of tree arcs too
        cp = rng.integers(0, N - 1, trail // 2)
        tail[N - 1 + n_red:N - 1 + n_red + cp.size] = tp[cp]
        head[N - 1 + n_red:N - 1 + n_red + cp.size] = tm[cp]
        assert korder[P] == last
    else:
        raise ValueError(family)
    return np.asarray(tail, np.int64), np.asarray(head, np.int64), np.asarray(korder, np.int64)


KR_FAMILIES = ["path_along", "path_against", "path_random", "star_hub0", "star_hubN", "loops_parallel",
               "forest", "complete_at_chunk_end", "complete_after_chunk_end"]
KR_NS = [2, 3, 1025, 8873, 8874, 12000, 16000, 16001, 262144, 262145]
KR_BIG = 1_000_003


def _kr_cases():
    out = []
    for N in KR_NS:
        for fam in KR_FAMILIES:
            out.append(pytest.param(N, fam, id=f"N{N}-{kr_variant(N)}-{fam}"))
    for fam in ("path_random", "star_hubN", "forest", "complete_after_chunk_end"):
        out.append(pytest.param(KR_BIG, fam, id=f"N{KR_BIG}-{kr_variant(KR_BIG)}-{fam}"))
    return out


def _run_kruskal(dev, korder_t, N, **kw):
    tree, n_tree = dev.kruskal(korder_t, N, **kw)
    nt = int(n_tree.item())
    return nt, tree[:nt].cpu().numpy()


def _check_forest(nt, got, ref):
    assert nt == ref.size
    assert np.array_equal(got, ref)
    assert (np.diff(got) > 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("N,family", _kr_cases())
def test_kruskal_matches_sequential_forest(dev, kr_tuning, N, family):
    """sx_kruskal == sequential Kruskal over the same order, under every first-chunk schedule."""
    import torch
    rng = np.random.default_rng(N + 7 * KR_FAMILIES.index(family))
    chunked = family.startswith("complete_")
    first = None
    for q in KR_QS:
        if chunked or first is None:
            tail, head, korder = kr_family(family, N, np.random.default_rng(rng.integers(1 << 31)), q)
            ref = orc.spanning_forest(korder, N, tail=tail, head=head)
            if family.startswith("forest"):
                assert ref.size < N - 1
            elif N > 1:
                assert ref.size == N - 1
            args = dict(tail=cu(tail, torch.int32), head=cu(head, torch.int32))
            kt = cu_korder(korder)
        kr_tuning(q)
        nt, got = _run_kruskal(dev, kt, N, **args)
        _check_forest(nt, got, ref)
        if not chunked:
            if first is None:
                first = got
            assert np.array_equal(got, first)


@pytest.mark.gpu
@pytest.mark.parametrize("S,D,n,complete", [
    pytest.param(40, 60, 49, False, id="N100-cta-smemlists-short"),
    pytest.param(40, 60, 1500, False, id="N100-cta-smemlists-row-missing"),
    pytest.param(30, 40, 1200, True, id="N70-cta-smemlists-whole-order"),
    pytest.param(5000, 7000, 30000, False, id="N12000-cta-globallists-row-missing"),
    pytest.param(10000, 10001, 60000, False, id="N20001-coop1-row-missing"),
    pytest.param(131073, 131072, 800000, False, id="N262145-coop4-prefix"),
])
def test_kruskal_ot_prefix(dev, kr_tuning, S, D, n, complete):
    """Implicit OT endpoints with `korder` a prefix (n < S D, ids anywhere below S D): the forest of the
    prefix, incomplete unless every arc is listed."""
    rng = np.random.default_rng(S + D + n)
    N = S + D
    if complete:
        korder = rng.permutation(S * D)
    else:
        lim = min((S - 1) * D, (1 << 32) - 1)                  # the last row (and maybe more) is never listed
        korder = np.unique(rng.integers(0, lim, 2 * n))[:n]
        korder = rng.permutation(korder)
    ref = orc.spanning_forest(korder, N, S=S, D=D)
    assert (ref.size == N - 1) == complete
    kt = cu_korder(korder)
    first = None
    for q in KR_QS:
        kr_tuning(q)
        nt, got = _run_kruskal(dev, kt, N, S=S, D=D)
        _check_forest(nt, got, ref)
        first = got if first is None else first
        assert np.array_equal(got, first)


# ==== tree potentials =====================================================================================
def _potentials_arc_list(dev, plus, minus, cost, N, root, plus_is_tail, rng):
    import torch
    from smart_crossover._native import SX_PLUS_IS_HEAD, SX_PLUS_IS_TAIL
    tail, head, ids = arc_list(plus, minus, plus_is_tail, rng)
    c = rng.random(tail.size) * 1e9                           # arcs outside the tree carry junk costs
    c[ids] = cost
    y = dev.tree_potentials(cu(ids), ids.size, N, cu(c), root, tail=cu(tail, torch.int32),
                            head=cu(head, torch.int32), plus=SX_PLUS_IS_TAIL if plus_is_tail else SX_PLUS_IS_HEAD)
    return y.cpu().numpy()


POT_NS = [2, 3, 2048, 2049, 2050]


@pytest.mark.gpu
@pytest.mark.parametrize("shape,N", [pytest.param(s, N, id=f"{s}-N{N}-{tour_path(N)}")
                                     for N in POT_NS for s in SHAPES])
def test_potentials_bit_exact_on_dyadic_costs(dev, shape, N):
    """Costs on a common dyadic grid: every sum the kernel forms is exact, so the potentials are bit-exact,
    for every root kind and both plus conventions."""
    rng = np.random.default_rng(N * 13 + SHAPES.index(shape))
    plus, minus = orient(*tree_shape(shape, N, rng), rng)
    cost = dyadic_costs(N - 1, rng)
    for kind in ROOTS:
        root = pick_root(kind, plus, minus, N, rng)
        m, E = exact_potentials(plus, minus, cost, N, root)
        want = grid_to_float(m, E)
        for plus_is_tail in (False, True):
            got = _potentials_arc_list(dev, plus, minus, cost, N, root, plus_is_tail, rng)
            assert got.tobytes() == want.tobytes(), (kind, plus_is_tail)


@pytest.mark.gpu
@pytest.mark.parametrize("shape,N", [
    pytest.param("path", 1 << 22, id="path-N4194304-coop"),
    pytest.param("path_shuffled", 1 << 20, id="path_shuffled-N1048576-coop"),
    pytest.param("recursive", 1 << 20, id="recursive-N1048576-coop"),
    pytest.param("binary", (1 << 20) - 1, id="binary-N1048575-coop"),
    pytest.param("star", 300001, id="star-N300001-coop"),
])
def test_potentials_bit_exact_large(dev, shape, N):
    """Deep and wide trees far past the single-CTA tour: bit-exact on dyadic costs from two roots."""
    rng = np.random.default_rng(N)
    plus, minus = orient(*tree_shape(shape, N, rng), rng)
    cost = dyadic_costs(N - 1, rng, span=20)
    for kind in ("last", "leaf"):
        root = pick_root(kind, plus, minus, N, rng)
        m, E = exact_potentials(plus, minus, cost, N, root)
        got = _potentials_arc_list(dev, plus, minus, cost, N, root, kind == "leaf", rng)
        assert got.tobytes() == grid_to_float(m, E).tobytes(), kind


OT_SHAPES = [(1, 1), (1, 2), (2, 1), (700, 1349), (700, 1350), (1500, 2500)]


def _ot_id(S, D):
    return f"ot{S}x{D}-N{S + D}-{tour_path(S + D)}"


@pytest.mark.gpu
@pytest.mark.parametrize("S,D", [pytest.param(S, D, id=_ot_id(S, D)) for S, D in OT_SHAPES])
def test_potentials_ot_padded_cost_matrix(dev, S, D):
    """Implicit OT arcs priced from a column slice of a wider matrix (ld > D): bit-exact on dyadic costs
    for every root kind."""
    rng = np.random.default_rng(S * D + 3)
    N = S + D
    tree, plus, minus = ot_tree(S, D, rng)
    ld, c0 = D + 37, 11
    Mfull = rng.random((S, ld)) * 1e9                          # junk outside the slice
    Mfull[:, c0:c0 + D] = dyadic_costs(S * D, rng).reshape(S, D)
    M = Mfull[:, c0:c0 + D]
    cost = M[tree // D, tree % D]
    Mt = cu(Mfull)
    for kind in ROOTS:
        root = pick_root(kind, plus, minus, N, rng)
        m, E = exact_potentials(plus, minus, cost, N, root)
        y = dev.tree_potentials(cu(tree), tree.size, N, Mt[:, c0:c0 + D], root, S=S, D=D, ld=ld)
        assert y.cpu().numpy().tobytes() == grid_to_float(m, E).tobytes(), kind
        # the same matrix packed (ld == D) gives the same bits
        y2 = dev.tree_potentials(cu(tree), tree.size, N, cu(np.ascontiguousarray(M)), root, S=S, D=D)
        assert y2.cpu().numpy().tobytes() == y.cpu().numpy().tobytes()


REAL_CASES = [("recursive", 2049), ("recursive", 2050), ("caterpillar", 20000), ("path_shuffled", 20000),
              ("broom", 100000), ("recursive", 400000)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape,N", [pytest.param(s, N, id=f"{s}-N{N}-{tour_path(N)}") for s, N in REAL_CASES])
def test_potentials_real_costs_normwise(dev, shape, N):
    """Real costs with mixed magnitudes (1% of them 1e6 times the rest) against the exact potentials.
    Normwise the error is below POT_ULPS_PER_ROUND * ceil(log2 H) * eps * max|y| (and so below the
    suite's 1e-9 * max|y|).  Elementwise, relative to each node's own |y|, it is not within 1e-9: the
    prefix sums of the tour carry the error of the expensive arcs to nodes with small potentials.  The
    count of such nodes is printed; it is the reason a double-double tour would be needed for an
    elementwise bar."""
    rng = np.random.default_rng(N + 1)
    plus, minus = orient(*tree_shape(shape, N, rng), rng)
    cost = mixed_costs(N - 1, rng)
    H = 2 * (N - 1)
    rounds = math.ceil(math.log2(H))
    for kind in ("last", "leaf"):
        root = pick_root(kind, plus, minus, N, rng)
        m, E = exact_potentials(plus, minus, cost, N, root)
        want = grid_to_float(m, E)
        got = _potentials_arc_list(dev, plus, minus, cost, N, root, False, rng)
        scale = np.abs(want).max()
        err = np.abs(got - want)
        assert err.max() <= 1e-9 * scale
        ulps = err.max() / (EPS * scale)
        n_rel = int((err > 1e-9 * np.abs(want)).sum())
        print(f"\n{shape} N={N} root={kind}: max err {ulps:.2f} eps*max|y| ({ulps / rounds:.3f} per round), "
              f"{n_rel} nodes beyond 1e-9 of their own |y|")
        assert ulps <= POT_ULPS_PER_ROUND * rounds


@pytest.mark.gpu
@pytest.mark.parametrize("N", [pytest.param(N, id=f"N{N}-{tour_path(N)}") for N in (6, 2049, 2050, 70000)])
def test_non_spanning_input_is_rejected(dev, N):
    """N - 1 arcs that are not a spanning tree (valid node ids only): a cycle plus an isolated node, an
    isolated root, a triangle plus a path (every node has an arc; the path is never reached from the root)
    and three parallel arcs with a path and two isolated nodes (every half-edge is reached from the root)
    all return SX_ERR_NOT_SPANNING, from both kernels."""
    import torch
    from smart_crossover._native import SX_ERR_NOT_SPANNING, SxError
    rng = np.random.default_rng(N)
    for name, plus, minus, root in non_spanning_cases(N):
        for plus_is_tail in (False, True):
            tail, head, ids = arc_list(plus, minus, plus_is_tail, rng)
            kw = dict(tail=cu(tail, torch.int32), head=cu(head, torch.int32), plus=int(plus_is_tail))
            with pytest.raises(SxError) as ei:
                dev.tree_potentials(cu(ids), ids.size, N, cu(rng.random(tail.size)), root, **kw)
            assert ei.value.code == SX_ERR_NOT_SPANNING, name
            with pytest.raises(SxError) as ei:
                dev.tree_flows(cu(ids), ids.size, N, cu(rng.random(N)), root, **kw)
            assert ei.value.code == SX_ERR_NOT_SPANNING, name
    # and a spanning tree right after, on the same sizes, is accepted
    plus, minus = orient(*tree_shape("recursive", N, rng), rng)
    cost = dyadic_costs(N - 1, rng)
    m, E = exact_potentials(plus, minus, cost, N, 0)
    assert _potentials_arc_list(dev, plus, minus, cost, N, 0, False, rng).tobytes() == grid_to_float(m, E).tobytes()


# ==== tree flows ==========================================================================================
def _flows_arc_list(dev, plus, minus, b, N, root, plus_is_tail, rng):
    import torch
    from smart_crossover._native import SX_PLUS_IS_HEAD, SX_PLUS_IS_TAIL
    tail, head, ids = arc_list(plus, minus, plus_is_tail, rng)
    f = dev.tree_flows(cu(ids), ids.size, N, cu(b), root, tail=cu(tail, torch.int32), head=cu(head, torch.int32),
                       plus=SX_PLUS_IS_TAIL if plus_is_tail else SX_PLUS_IS_HEAD)
    return f.cpu().numpy()


# N = 2050 and 1026 put H just above a multiple of 1024 (uneven chunks, empty threads in flow_scan_kernel);
# N = 300 leaves most of its 1024 threads empty
FLOW_CASES = [("path", 2), ("star", 3), ("recursive", 300), ("broom", 1026), ("caterpillar", 2048),
              ("recursive", 2049), ("recursive", 2050), ("path_shuffled", 2050), ("star", 2050),
              ("binary", 2050), ("path_reversed", 2050), ("recursive", 40000), ("path_shuffled", 100000)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape,N", [pytest.param(s, N, id=f"{s}-N{N}-{tour_path(N)}") for s, N in FLOW_CASES])
def test_tree_flows_wide_supplies(dev, shape, N):
    """Supplies spread over 1e-6 .. 1e6 with random signs, Sum b != 0, every root kind, both plus
    conventions: every flow within 1 ulp of the exact subtree sum where sum|b| / |sum| <= 2^50 / H, and
    within 1/2 ulp + 2^-103 H sum|b| everywhere."""
    rng = np.random.default_rng(N * 3 + len(shape))
    plus, minus = orient(*tree_shape(shape, N, rng), rng)
    b = wide_supplies(N, rng)
    H = 2 * (N - 1)
    for kind in ROOTS:
        root = pick_root(kind, plus, minus, N, rng)
        m, E = exact_subtree_flows(plus, minus, b, N, root)
        abs_b = float(np.abs(np.delete(b, root)).sum())
        for plus_is_tail in (False, True):
            got = _flows_arc_list(dev, plus, minus, b, N, root, plus_is_tail, rng)
            one, gen, rule, exact = flow_bounds(m, E, got, H, abs_b)
            assert one[rule].all(), (kind, plus_is_tail, np.flatnonzero(rule & ~one)[:5])
            assert gen.all(), (kind, plus_is_tail)


def zero_sum_supplies(plus, minus, N, root, rng):
    """Dyadic supplies at two far-apart scales (k * 2^30 and k * 2^-30, k < 2^12), paired off (x, -x) inside
    the subtrees of about a quarter of the nodes so that those subtrees sum to exactly 0.  The tour's
    running sums need about 90 bits: exact in a double-double, not in a double."""
    order, child, plus_child = tree_bfs(plus, minus, N, root)
    par = np.arange(N)
    par[child] = np.where(plus_child, minus, plus)
    kids = [[] for _ in range(N)]
    for v in order[1:].tolist():
        kids[par[v]].append(v)

    def value():
        return float(rng.integers(1, 1 << 12)) * (2.0 ** 30 if rng.random() < 0.5 else 2.0 ** -30)
    b = np.zeros(N)
    zero_roots = set(rng.choice(np.delete(np.arange(N), root), max(1, N // 4), replace=False).tolist())
    unpaired = [None] * N                     # nodes of v's subtree whose supply is not set yet
    for v in order[::-1].tolist():            # children before parents
        pool = [v]
        for u in kids[v]:
            pool.extend(unpaired[u])
            unpaired[u] = None
        if v in zero_roots:
            rng.shuffle(pool)
            if len(pool) % 2:
                b[pool.pop()] = 0.0
            for a_, c_ in zip(pool[0::2], pool[1::2]):
                x = value()
                b[a_], b[c_] = x, -x
            pool = []
        unpaired[v] = pool
    for v in unpaired[root]:
        b[v] = value() * (1 if rng.random() < 0.5 else -1)
    return b, sorted(zero_roots)


@pytest.mark.gpu
@pytest.mark.parametrize("shape,N", [pytest.param(s, N, id=f"{s}-N{N}-{tour_path(N)}")
                                     for s, N in (("recursive", 2049), ("caterpillar", 2050), ("binary", 9000))])
def test_tree_flows_exact_zeros(dev, shape, N):
    """Subtrees whose supplies cancel exactly give a flow of +-0.0, never a tiny negative (which would
    start a spurious push); every other flow is exact too (the sums fit in a double-double)."""
    rng = np.random.default_rng(N + 99)
    plus, minus = orient(*tree_shape(shape, N, rng), rng)
    root = pick_root("leaf", plus, minus, N, rng)
    b, zero_roots = zero_sum_supplies(plus, minus, N, root, rng)
    m, E = exact_subtree_flows(plus, minus, b, N, root)
    want = grid_to_float(m, E)
    n_zero = int((np.array([v == 0 for v in m])).sum())
    assert n_zero >= len(zero_roots)
    for plus_is_tail in (False, True):
        got = _flows_arc_list(dev, plus, minus, b, N, root, plus_is_tail, rng)
        assert np.array_equal(got, want)                      # == treats -0.0 as 0.0
        assert (got[want == 0] == 0).all()


@pytest.mark.gpu
def test_tree_flows_large_path_integer_supplies(dev):
    """A path of 2^22 nodes (the deepest tour) rooted in the middle, integer supplies: the flows are the
    exact prefix / suffix sums."""
    N = 1 << 22
    rng = np.random.default_rng(22)
    b = rng.integers(-(1 << 20), 1 << 20, N).astype(np.float64)
    root = N // 3
    i = np.arange(N - 1)
    plus, minus = i + 1, i                                    # arc i: i -> i+1, +1 at i+1
    pre = np.cumsum(b.astype(np.int64))
    suf = np.cumsum(b[::-1].astype(np.int64))[::-1]
    # arcs left of the root hang their subtree 0..i at the minus end; right of it, i+1..N-1 at the plus end
    want = np.where(i < root, -pre[np.minimum(i, N - 1)], suf[np.minimum(i + 1, N - 1)]).astype(np.float64)
    for plus_is_tail in (False, True):
        got = _flows_arc_list(dev, plus, minus, b, N, root, plus_is_tail, rng)
        assert np.array_equal(got, want), plus_is_tail


@pytest.mark.gpu
@pytest.mark.parametrize("S,D", [pytest.param(S, D, id=_ot_id(S, D)) for S, D in ((3, 2), (700, 1350), (1200, 1800))])
def test_tree_flows_ot_zero_flows_drive_the_same_push(dev, S, D):
    """An OT tree whose flows are chosen first, 30% of them exactly 0 and the rest positive (dyadic, at 2^16
    and 2^-16 scales), with the supplies that make them the solution.  The device flows equal them bit for
    bit (zeros as +-0.0, for two roots and unbalanced supplies), and the push phase from the device flows
    returns the same basis and push count as from the exact flows.  A tiny negative in place of a zero
    would make the push phase assert or push."""
    from smart_crossover.formats import OptTransport
    from smart_crossover.network_methods.net_manager import OTManager
    from smart_crossover.network_methods.tree_BI import push_tree_to_bfs
    rng = np.random.default_rng(S + D)
    N = S + D
    tree, plus, minus = ot_tree(S, D, rng)
    T = tree.size
    mag = rng.integers(1, 1 << 12, T) * np.where(rng.random(T) < 0.5, 2.0 ** 16, 2.0 ** -16)
    x = np.where(rng.random(T) < 0.3, 0.0, mag)
    b = np.zeros(N)
    np.add.at(b, plus, x)                                     # b = A x: few arcs per node, 44-bit span: exact
    np.add.at(b, minus, -x)
    xm, E = to_grid(x)
    b_ints = [0] * N
    for p, q, v in zip(plus.tolist(), minus.tolist(), xm.tolist()):
        b_ints[p] += int(v)
        b_ints[q] -= int(v)
    assert np.array_equal(b, grid_to_float(b_ints, E)), "supplies not exact"
    b[N - 1] += 1.0                                           # unbalanced: the root's row is dropped
    for root in (N - 1, 0):
        m, E2 = exact_subtree_flows(plus, minus, b, N, root)
        want = grid_to_float(m, E2)
        if root == N - 1:
            assert np.array_equal(want, x)
        got = dev.tree_flows(cu(tree), T, N, cu(b), root, S=S, D=D).cpu().numpy()
        assert np.array_equal(got, want)
        assert (got[want == 0] == 0).all()
    got = dev.tree_flows(cu(tree), T, N, cu(b), N - 1, S=S, D=D).cpu().numpy()
    vb_ref, it_ref = orc.push_tree_to_bfs(tree, x, S, D)
    ot = OptTransport(np.full(S, float(D)), np.full(D, float(S)), rng.random((S, D)))   # the push reads S, D
    vb, it = push_tree_to_bfs(OTManager(ot), tree, _flows=got)
    assert it == it_ref
    assert np.array_equal(vb.astype(np.int64), vb_ref)

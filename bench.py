#!/usr/bin/env python
"""bench.py -- headline benchmark of the network-crossover hot path on B200.

Metric (BASELINE.json): OT arcs priced/s (with % of the HBM roofline) + tree-basis build ms.
Workload: dense synthetic OT 60 000 x 60 000 (3.6e9 arcs, 28.8 GB fp64 cost; BASELINE.json
configs[4], the largest configuration the metric is quoted on and it fits one 180 GB GPU),
row-sharded over N ranks (strong scaling: the matrix is fixed, each rank prices S/N rows).
A "step" is one column-generation pricing pass over the whole matrix: reduced costs of every
arc against the duals, violator count, min reduced cost and the global top-K most violating
arcs (NCCL all-gather + merge when N > 1).

    python bench.py --gpus 1 --steps 200 --warmup 10
    python -m torch.distributed.run --nproc-per-node 8 ... bench.py --gpus 8 ...
    python bench.py --impl reference ...        # CPU arm: the oracle port on all host cores

`value`   : arcs/s with everything resident in HBM (duals included), device-timed.
`e2e`     : the same pass through the public call (`ShardedDensePricer.price`) with the duals in
            pinned host memory: H2D of y and D2H of (count, min, top-K) inside every step.
            The cost matrix is uploaded once per problem (manager state, like `ot.M` in the
            reference's `OTManager`), not per pricing pass; `e2e_cold` adds that upload.
`roofline`: achieved HBM GB/s of the pricing kernel alone (8 B per arc / CUDA-event time).

`--dump-outputs DIR` writes the result of the last timed step (what `PriceResult` hands a caller: violator
count, min reduced cost, top-K arc ids and reduced costs) as DIR/<name>.npy, float64, and for the second leg as
DIR/c4_<name>.npy.  The inputs are generated from fixed seeds, so two builds run with the same arguments can be
compared file for file.  With `--impl reference` the dump fixes the host's row sample at the first 512 seeded rows
instead of sizing it from a timed pass.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "smart-crossover_b200"), os.path.join(ROOT, "tests", "golden")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

METRIC = "ot_arcs_priced_per_s"
UNIT = "arcs/s"
TOL = 1e-6


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--size", type=int, default=60000, help="S = D of the dense OT instance")
    ap.add_argument("--rows", type=int, default=0, help="S if different from --size (profiling a per-rank slab shape)")
    ap.add_argument("--topk", type=int, default=1024)
    ap.add_argument("--variant", type=int, default=-1, help="-1 auto (TMA), 0 TMA, 1 vector loads, 2 scalar loads")
    ap.add_argument("--violators", type=float, default=1e-4, help="target fraction of violating arcs")
    ap.add_argument("--no-tree", action="store_true", help="skip the tree-basis build timings")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--exchange", default="ll", choices=["ll", "p2p", "nccl"],
                    help="N > 1: exchange of the result blocks: NVLink flag-in-data stores polled by the merge "
                         "kernel (default), peer stores + flag + wait kernel, or NCCL all-gather")
    ap.add_argument("--no-fused", action="store_true",
                    help="price / select / push as separate launches (round-1 path) instead of the fused kernel")
    ap.add_argument("--no-c4", action="store_true", help="skip the second leg (dense OT 20 000 x 20 000)")
    ap.add_argument("--no-manager", action="store_true", help="skip the OTManager end-to-end leg")
    ap.add_argument("--no-balance", action="store_true",
                    help="N > 1: equal row shards instead of shards sized by each GPU's measured rate")
    ap.add_argument("--c4-size", type=int, default=20000)
    ap.add_argument("--sweep", action="store_true", help="time every pricing-kernel variant / tuning and exit")
    ap.add_argument("--sweep-ab", default="", metavar="I,J,..",
                    help="with --sweep: interleaved A/B timing of these TMA shape indices only")
    ap.add_argument("--score-ctas", type=int, default=0, help="sx_score_set_tuning (3 or 4 resident CTAs per SM)")
    ap.add_argument("--kruskal-chunk", type=int, default=0, help="sx_kruskal_set_tuning (first chunk in quarters of N)")
    ap.add_argument("--tree-only", type=int, default=0, metavar="S",
                    help="only time the tree-basis build on an S x S instance and exit")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the result of the last timed pricing step to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.sweep or args.tree_only):
        ap.error("--dump-outputs needs a pricing run (not --sweep or --tree-only)")
    return args


DUMP_MAX_TOPK = 1 << 20      # top-K entries written per leg: at most 3 x 8 MB, both legs within 64 MB


def dump_outputs(out_dir, prefix, count, min_rc, ids, rc):
    """Writes one pricing result, as `device.PriceResult` returns it, to out_dir/<prefix><name>.npy in float64
    (arc ids are exact below 2^53).  A top-K list longer than DUMP_MAX_TOPK is cut to a fixed, seeded sample of
    its positions, which are written as <prefix>topk_pos.npy."""
    os.makedirs(out_dir, exist_ok=True)
    ids, rc = np.asarray(ids), np.asarray(rc)
    arrays = {"n_violating": [count], "min_rc": [min_rc]}
    if ids.size > DUMP_MAX_TOPK:
        pos = np.sort(np.random.default_rng(0).choice(ids.size, DUMP_MAX_TOPK, replace=False))
        ids, rc = ids[pos], rc[pos]
        arrays["topk_pos"] = pos
    arrays["topk_id"], arrays["topk_rc"] = ids, rc
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), np.asarray(a, dtype=np.float64))


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json, copy read+write)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.proc = None
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                c = [x.strip() for x in line.split(",")]
                if len(c) < 7:
                    continue
                try:
                    sm.append(float(c[0])); mx.append(float(c[1]))
                except ValueError:
                    continue
                for nm, v in zip(names, c[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), samples=len(sm))
        out["reasons"] = sorted(reasons)
        return out


# ------------------------------------------------------------------------------------------------
# synthetic instance (SURVEY.md section 8d): squared-Euclidean cost between uniform points, planted duals
# ------------------------------------------------------------------------------------------------
def make_points(S, D, device, seed=20260005):
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    P = torch.rand(S, 2, generator=g, device=device, dtype=torch.float64)
    Q = torch.rand(D, 2, generator=g, device=device, dtype=torch.float64)
    a = torch.rand(S, generator=g, device=device, dtype=torch.float64)
    return P, Q, a


def cost_rows(P, Q, r0, r1):
    dx = P[r0:r1, 0:1] - Q[None, :, 0]
    dy = P[r0:r1, 1:2] - Q[None, :, 1]
    return dx * dx + dy * dy


def make_slab(P, Q, row0, S_loc, out=None, block=1000):
    import torch
    D = Q.shape[0]
    M = out if out is not None else torch.empty(S_loc, D, dtype=torch.float64, device=P.device)
    for r in range(0, S_loc, block):
        e = min(S_loc, r + block)
        M[r:e] = cost_rows(P, Q, row0 + r, row0 + e)
    return M


def planted_duals(P, Q, a, M_loc, row0, frac, world, sample_rows=1500):
    """Planted duals plus noise (SURVEY.md section 8d): y0 = (a, b) with b_j = min_i (M_ij + a_i) makes
    every reduced cost >= 0 and tight once per column; y = y0 + sigma * N(0, 1) on every node, with
    sigma bisected on a row sample so that about `frac` of the arcs end up with rc < -tol.  The same
    seeded noise on every rank."""
    import torch
    import torch.distributed as dist
    S_loc, D = M_loc.shape
    S = P.shape[0]
    b = torch.full((D,), float("inf"), dtype=torch.float64, device=M_loc.device)
    for r in range(0, S_loc, 1000):
        e = min(S_loc, r + 1000)
        b = torch.minimum(b, (M_loc[r:e] + a[row0 + r:row0 + e, None]).min(dim=0).values)
    if world > 1:
        dist.all_reduce(b, op=dist.ReduceOp.MIN)
    if frac <= 0:
        return torch.cat([a, b - 1e-3])
    g = torch.Generator(device=M_loc.device).manual_seed(20260105)
    noise = torch.randn(S + D, generator=g, device=M_loc.device, dtype=torch.float64)
    R = min(sample_rows, S)
    rc0 = cost_rows(P, Q, 0, R) - (b[None, :] - a[:R, None])       # same rows on every rank
    dn = noise[S:][None, :] - noise[:R, None]                      # rc = rc0 - sigma * dn
    lo, hi = 0.0, 1.0
    for _ in range(40):
        mid = 0.5 * (lo + hi)
        f = float((rc0 - mid * dn < -TOL).sum().item()) / rc0.numel()
        lo, hi = (mid, hi) if f < frac else (lo, mid)
    return torch.cat([a, b]) + hi * noise


# ------------------------------------------------------------------------------------------------
# CPU legs (oracle port): cpu_baseline (1 thread, rank 0) and --impl reference (all host threads)
# ------------------------------------------------------------------------------------------------
def cpu_price_rate(M_h, y_h, K, threads, reps):
    from oracle import network_oracle as orc
    best = None
    for _ in range(reps):
        t0 = time.perf_counter()
        orc.price_dense_ot_blocked(M_h, y_h, K, TOL, threads=threads, block_rows=64)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return M_h.size / best, best


def run_reference(args):
    """Reference arm: the reference's pricing pass (`c - A.T @ y`, `np.all(rc >= -tol)`,
    net_manager.py:474-497) as restated by the oracle (bitwise-equal dense form, SURVEY.md H4),
    on all host threads, over a bounded row sample of the same 60 000-column instance."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    S = D = args.size
    threads = os.cpu_count() or 1
    rng = np.random.default_rng(20260005)
    rows = 512
    Q = rng.random((D, 2)); P = rng.random((rows, 2)); a = rng.random(rows)
    M = (P[:, 0:1] - Q[None, :, 0]) ** 2 + (P[:, 1:2] - Q[None, :, 1]) ** 2
    b = (M + a[:, None]).min(axis=0) + 2e-3
    y = np.concatenate([a, b])
    if args.dump_outputs:
        # a dumped result must not depend on how fast this host is: the first seeded rows, not a timed size
        rows2 = min(S, rows)
    else:
        # size the per-step sample so that steps + warmup take about two minutes
        rate, dt = cpu_price_rate(M, y, args.topk, threads, 1)
        budget = 120.0 / max(1, args.steps + args.warmup)
        rows2 = int(min(S, max(256, rows * budget / dt)))
        rows2 = min(rows2, 8192)
    if rows2 != rows:
        P = rng.random((rows2, 2)); a = rng.random(rows2)
        M = (P[:, 0:1] - Q[None, :, 0]) ** 2 + (P[:, 1:2] - Q[None, :, 1]) ** 2
        b = (M + a[:, None]).min(axis=0) + 2e-3
        y = np.concatenate([a, b])
    from oracle import network_oracle as orc
    for _ in range(args.warmup):
        orc.price_dense_ot_blocked(M, y, args.topk, TOL, threads=threads, block_rows=64)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        result = orc.price_dense_ot_blocked(M, y, args.topk, TOL, threads=threads, block_rows=64)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, "", *result)
    value = M.size * args.steps / dt
    sample = f"{rows2} of {S} rows x {D} cols per step ({M.size:.3g} arcs), oracle port, NumPy row blocks"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": f"dense synthetic OT {S}x{D} ({S * D:.3g} arcs, {8 * S * D / 1e9:.1f} GB fp64 cost) "
                                   f"column-generation pricing pass, host CPU on a bounded row sample per step",
                       "S": S, "D": D, "topk": args.topk, "tol": TOL, "rows_per_step": rows2},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# tree-basis build timing (single GPU): scores -> argsort -> Kruskal order -> tree -> potentials
# ------------------------------------------------------------------------------------------------
def cpu_tree_build_ot(x, s, d, M, S, D, note):
    """Oracle port of the same steps on ONE host core: scores (net_manager.py:377-378), stable argsort
    (:379), Kruskal on the stable order of -w (tree_BI.py:47-57), potentials of the tree (B^T y = c_B)."""
    from oracle import network_oracle as orc
    t = [time.perf_counter()]
    F = orc.ot_flow_scores(x, s, d); t.append(time.perf_counter())
    q = orc.stable_queue(F); t.append(time.perf_counter())
    tree = orc.max_weight_spanning_tree(F, S, D, drop_zero_weight=False); t.append(time.perf_counter())
    orc.ot_tree_potentials(tree, M); t.append(time.perf_counter())
    names = ["score", "argsort", "kruskal (incl. its own stable argsort)", "potentials"]
    return {"ms": round(1e3 * (t[-1] - t[0]), 2), "breakdown_ms": {n: round(1e3 * (t[i + 1] - t[i]), 2) for i, n in enumerate(names)},
            "cores": 1, "kind": "port", "host_cpus": os.cpu_count(), "sample": note}


def time_tree_build(S, D, device, reps=3, cpu=None, call_host=False):
    """`cpu`: None = no CPU leg; (S_cpu, D_cpu) = time the oracle port on an instance of that shape (the same
    instance when equal to (S, D), else a smaller stand-in built the same way)."""
    import torch
    from smart_crossover import device as dev
    P, Q, a = make_points(S, D, device, seed=20260002)
    M = make_slab(P, Q, 0, S)
    g = torch.Generator(device=device).manual_seed(99)
    s = torch.rand(S, generator=g, device=device, dtype=torch.float64) + 0.1
    d = torch.rand(D, generator=g, device=device, dtype=torch.float64) + 0.1
    s /= s.sum(); d /= d.sum()
    t = 1.0 + 40.0 * (M / 0.33)
    x = ((s[:, None] * d[None, :]) / (t * t * t * t)).reshape(-1)
    x *= 1.0 + 1e-3 * torch.rand(x.shape, generator=g, device=device, dtype=torch.float64)
    del t
    N = S + D
    nt = N - 1
    # (A) tree-basis build as tree_BI.tree_basis_identify runs it: scores -> head of the Kruskal order
    #     (sx_kruskal_prefix, 16 N arcs) -> union-find -> potentials
    best = None
    for _ in range(reps + 1):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        ev[0].record()
        F, hist = dev.score_ot(x, s, d, want_hist=True)
        ev[1].record()
        head = dev.kruskal_prefix(F, 16 * N, hist=hist)
        ev[2].record()
        tree, n_tree = dev.kruskal(head, N, S=S, D=D)
        ev[3].record()
        y = dev.tree_potentials(tree, nt, N, M, N - 1, S=S, D=D)
        ev[4].record()
        torch.cuda.synchronize()
        parts = [ev[i].elapsed_time(ev[i + 1]) for i in range(4)]
        assert head is not None and int(n_tree.item()) == nt
        if best is None or sum(parts) < sum(best):
            best = parts
        tree_a = tree.clone()
        del F, head, tree, y
    # (B) the full sorted queue of get_sorted_flows (every arc ranked) and the tree from that order
    full = None
    for _ in range(reps + 1):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
        ev[0].record()
        F = dev.score_ot(x, s, d)
        ev[1].record()
        order, skey = dev.argsort_f64(F)
        ev[2].record()
        from smart_crossover.network_methods.tree_BI import PREFIX_MIN_ARCS
        korder = dev.kruskal_order_head(skey, order, 16 * N) if S * D >= PREFIX_MIN_ARCS else None   # as tree_BI does
        if korder is None:
            korder = dev.kruskal_order(skey, order)
        ev[3].record()
        tree, n_tree = dev.kruskal(korder, N, S=S, D=D)
        ev[4].record()
        y = dev.tree_potentials(tree, nt, N, M, N - 1, S=S, D=D)
        ev[5].record()
        torch.cuda.synchronize()
        parts = [ev[i].elapsed_time(ev[i + 1]) for i in range(5)]
        assert int(n_tree.item()) == nt and bool((tree == tree_a).all())      # same tree either way
        if full is None or sum(parts) < sum(full):
            full = parts
        del F, order, skey, korder, tree, y
    # the reference-facing call with HOST arrays in and out (net_manager.py:368-379): upload of x, scores, sort,
    # download of the two n-sized results through pinned staging (wall clock, once)
    call_s = None
    if call_host:
        from smart_crossover.formats import OptTransport
        from smart_crossover.network_methods.net_manager import OTManager
        x_h, s_h, d_h = x.cpu().numpy(), s.cpu().numpy(), d.cpu().numpy()
        mgr = OTManager(OptTransport(s_h, d_h, np.zeros((1, 1))))            # the cost matrix plays no part in this call
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        q_h, sc_h = mgr.get_sorted_flows(x_h)
        call_s = time.perf_counter() - t0
        assert q_h.shape == (S * D,) and sc_h.shape == (S * D,)
        del q_h, sc_h, x_h, mgr
    names = ["score", "kruskal_prefix", "kruskal", "potentials"]
    names_full = ["score", "argsort", "kruskal_order", "kruskal", "potentials"]
    from smart_crossover.network_methods.tree_BI import use_prefix_path
    prefix = use_prefix_path(S * D, N)                      # what tree_basis_identify runs on bare weights
    cpu_leg = None
    if cpu is not None:
        if tuple(cpu) == (S, D):
            cpu_leg = cpu_tree_build_ot(x.cpu().numpy(), s.cpu().numpy(), d.cpu().numpy(), M.cpu().numpy(), S, D,
                                        "the same instance, copied to the host")
        else:
            Sc, Dc = cpu
            Pc, Qc, _ = make_points(Sc, Dc, device, seed=20260002)
            Mc = make_slab(Pc, Qc, 0, Sc)
            gc_ = torch.Generator(device=device).manual_seed(99)
            sc = torch.rand(Sc, generator=gc_, device=device, dtype=torch.float64) + 0.1
            dc = torch.rand(Dc, generator=gc_, device=device, dtype=torch.float64) + 0.1
            sc /= sc.sum(); dc /= dc.sum()
            tc = 1.0 + 40.0 * (Mc / 0.33)
            xc = ((sc[:, None] * dc[None, :]) / (tc * tc * tc * tc)).reshape(-1)
            cpu_leg = cpu_tree_build_ot(xc.cpu().numpy(), sc.cpu().numpy(), dc.cpu().numpy(), Mc.cpu().numpy(), Sc, Dc,
                                        f"stand-in {Sc}x{Dc} ({Sc * Dc} arcs) built like the {S}x{D} instance: the "
                                        f"full-size oracle run takes minutes (SURVEY.md section 8d)")
            cpu_leg["arcs"] = Sc * Dc
    return {"workload": f"OT {S}x{D} ({S * D} arcs)", "ms": round(sum(best) if prefix else sum(full), 4),
            "cpu_baseline": cpu_leg, "get_sorted_flows_host_call_s": None if call_s is None else round(call_s, 4),
            "path": "kruskal_prefix" if prefix else "full_argsort",
            "kruskal_prefix_ms": round(sum(best), 4),
            "breakdown_ms": {n: round(v, 4) for n, v in zip(names, best)},
            "with_full_argsort_ms": round(sum(full), 4),
            "with_full_argsort_breakdown_ms": {n: round(v, 4) for n, v in zip(names_full, full)}}


def time_price_arcs_planted(N, E, device, frac=1e-4, reps=20):
    """`price_arcs_kernel` (17 B per arc: c 8 + tail 4 + head 4 + status 1; y gathers from L2) on planted
    near-optimal duals: c_k = (y_tail - y_head) + slack_k with slack >= 0, and `frac` of the arcs pushed below
    -tol -- the converged regime a column-generation pass sees, not the 44 % violators of the flow-score tree."""
    import torch
    from smart_crossover import device as dev
    g = torch.Generator(device=device).manual_seed(20260303)
    tail = torch.randint(0, N, (E,), generator=g, device=device, dtype=torch.int32)
    head = (tail + 1 + torch.randint(0, N - 1, (E,), generator=g, device=device, dtype=torch.int32)) % N
    y = torch.rand(N, generator=g, device=device, dtype=torch.float64) * 100.0
    slack = torch.rand(E, generator=g, device=device, dtype=torch.float64) + 1e-3
    viol = torch.rand(E, generator=g, device=device, dtype=torch.float64) < frac
    slack = torch.where(viol, -slack, slack)
    c = (y[tail.long()] - y[head.long()]) + slack
    del slack
    vb = torch.full((E,), -1, dtype=torch.int8, device=device)
    pr = dev.Pricer(device, 1024, fused=False)
    for _ in range(3):
        pr.reset(); pr.price_arcs(c, tail, head, vb, y)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        pr.reset()
        a.record()
        pr.price_arcs(c, tail, head, vb, y)
        b.record()
    pr.select()
    torch.cuda.synchronize()
    res = pr.fetch()
    ms = float(np.median([a.elapsed_time(b) for a, b in ev]))
    exact = int(((c - (y[tail.long()] - y[head.long()])) < -TOL).sum().item())
    assert res.n_violating == exact, (res.n_violating, exact)
    peak, _ = measured_peak_gbs()
    gbs = 17.0 * E / (ms * 1e-3) / 1e9
    return {"arcs": E, "nodes": N, "violating_arcs": res.n_violating, "kernel_ms": round(ms, 4),
            "arcs_per_s": E / (ms * 1e-3), "algorithmic_bytes_per_arc": 17, "achieved_GBs": round(gbs, 1),
            "frac_of_measured_peak": round(gbs / peak, 4),
            "l2": f"inputs {17 * E / 1e6:.0f} MB vs 126 MB L2" + (" (L2-resident between repetitions)" if 17 * E < 1.2e8 else "")}


def time_sinkhorn(S, D, device, iters=20):
    """The device Sinkhorn warm start (`sx_sinkhorn_ot`; the reference's driver calls POT for it,
    scripts/run_network_crossover.py:96): ms per Sinkhorn-Knopp iteration = two streaming passes over the fp64
    cost matrix (column log-sum-exp, row log-sum-exp), 16 B per arc and iteration.  Parity of this function is
    UNPINNED (POT is not installed anywhere reachable): its oracle restates POT's published loop."""
    import ctypes
    import torch
    from smart_crossover import device as dev
    from smart_crossover._native import check, lib
    P, Q, a = make_points(S, D, device, seed=20260004)
    M = make_slab(P, Q, 0, S)
    g_ = torch.Generator(device=device).manual_seed(5)
    sa = torch.rand(S, generator=g_, device=device, dtype=torch.float64) + 0.1
    sb = torch.rand(D, generator=g_, device=device, dtype=torch.float64) + 0.1
    sa /= sa.sum(); sb /= sb.sum()
    f = torch.empty(S, dtype=torch.float64, device=device)
    gg = torch.empty(D, dtype=torch.float64, device=device)
    ws = dev._ws(lib.sx_sinkhorn_workspace_bytes(S, D), device)
    it_h, err_h = ctypes.c_int64(0), ctypes.c_double(0.0)
    reg = 0.01 * float(M[:64].median().item())

    def run(n):
        check(lib.sx_sinkhorn_ot(dev._ptr(M), M.stride(0), S, D, dev._ptr(sa), dev._ptr(sb), reg, n, 0.0, 10, dev._ptr(f),
                                 dev._ptr(gg), None, ctypes.byref(it_h), ctypes.byref(err_h), dev._ptr(ws), ws.numel(),
                                 dev._stream()), "sx_sinkhorn_ot")
    run(3)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run(iters)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    peak, _ = measured_peak_gbs()
    gbs = 16.0 * S * D / (ms * 1e-3) / 1e9
    ok = bool(torch.isfinite(f).all().item() and torch.isfinite(gg).all().item())
    return {"workload": f"log-domain Sinkhorn-Knopp on OT {S}x{D}, reg = 0.01 median(M)", "ms_per_iteration": round(ms, 4),
            "iterations_timed": iters, "algorithmic_bytes_per_arc_and_iteration": 16, "achieved_GBs": round(gbs, 1),
            "frac_of_measured_peak": round(gbs / peak, 4), "finite": ok,
            "parity": "unpinned: POT (third party, scripts/run_network_crossover.py:96) is not installed; the oracle "
                      "restates its published Sinkhorn-Knopp loop and the device plan matches it to 1e-9"}


def cpu_mcf_path(tail, head, c, u, x, A, N):
    """Oracle port on ONE host core: MCF flow indicators (net_manager.py:156-182), stable argsort (:184),
    Kruskal over the stable order of -w, potentials of the forest's tree."""
    from oracle import network_oracle as orc
    t = [time.perf_counter()]
    ind = orc.mcf_flow_scores(x, u, A); t.append(time.perf_counter())
    orc.stable_queue(ind); t.append(time.perf_counter())
    tree = orc.spanning_forest(orc.kruskal_order(ind), N, tail=tail, head=head); t.append(time.perf_counter())
    if tree.size == N - 1:
        orc.tree_potentials(tail[tree], head[tree], c[tree], N, N - 1)
    t.append(time.perf_counter())
    names = ["score", "argsort", "kruskal (incl. its own stable argsort)", "potentials"]
    return {"ms": round(1e3 * (t[-1] - t[0]), 1), "breakdown_ms": {n: round(1e3 * (t[i + 1] - t[i]), 1) for i, n in enumerate(names)},
            "cores": 1, "kind": "port", "host_cpus": os.cpu_count(), "sample": "the same instance (built on the host)"}


def time_mcf_path(N, E, device, reps=3, cpu=False):
    """BASELINE.json configs[2] shape (NETGEN-style 1M nodes / 10M arcs): scoring, sort, spanning
    forest, potentials and arc pricing on one GPU, CUDA-event times (best of `reps`)."""
    import scipy.sparse as sp
    import torch
    import cases
    from smart_crossover import device as dev
    tail, head, b, c, u = cases.netgen_like(N, E, 20260003)
    x = cases.mcf_interior_flow(u, 20260003)
    A = sp.csr_matrix((np.concatenate([np.ones(E, np.int8), -np.ones(E, np.int8)]),
                       (np.concatenate([tail, head]), np.concatenate([np.arange(E)] * 2))), shape=(N, E))
    A.sort_indices()
    cu = lambda a, dt=None: (torch.from_numpy(np.ascontiguousarray(a)).to(dt) if dt else
                             torch.from_numpy(np.ascontiguousarray(a))).to(device)
    t32, h32 = cu(tail, torch.int32), cu(head, torch.int32)
    xs, us, cs = cu(x), cu(u), cu(c)
    ptr, arc, sgn = cu(A.indptr, torch.int64), cu(A.indices, torch.int32), cu(A.data, torch.int8)
    vb = cu(np.where(x > u / 2, -2, -1).astype(np.int8))
    best = None
    pr = dev.Pricer(device, 1024)                           # buffers of the pricing pass: allocated once per problem
    for _ in range(reps + 1):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(8)]
        ev[0].record()
        ind = dev.score_mcf(xs, us, t32, h32, ptr, arc, sgn)
        ev[1].record()
        order, skey = dev.argsort_f64(ind)
        ev[2].record()
        korder = dev.kruskal_order(skey, order)
        ev[3].record()
        tree, n_tree = dev.kruskal(korder, N, tail=t32, head=h32)
        ev[4].record()
        y = dev.tree_potentials(tree, N - 1, N, cs, N - 1, tail=t32, head=h32, plus=1)
        ev[5].record()
        pr.reset(); pr.price_arcs(cs, t32, h32, vb, y)
        ev[6].record()
        pr.select()
        ev[7].record()
        torch.cuda.synchronize()
        parts = [ev[i].elapsed_time(ev[i + 1]) for i in range(7)]
        if best is None or sum(parts) < sum(best):
            best = parts
    res = pr.fetch()
    names = ["score", "argsort", "kruskal_order", "kruskal", "potentials", "price_arcs", "topk"]
    cpu_leg = cpu_mcf_path(tail, head, c, u, x, A.astype(np.float64), N) if cpu else None
    del xs, us, cs, t32, h32, ptr, arc, sgn, vb
    torch.cuda.empty_cache()
    planted = [time_price_arcs_planted(N, E, device), time_price_arcs_planted(10 * N, 10 * E, device, reps=10)]
    return {"workload": f"NETGEN-style MCF {N} nodes / {E} arcs", "tree_build_ms": round(sum(best[:5]), 4),
            "breakdown_ms": {n: round(v, 4) for n, v in zip(names, best)}, "cpu_baseline": cpu_leg,
            "price_arcs_per_s": E / ((best[5] + best[6]) * 1e-3), "violating_arcs": res.n_violating,
            "price_arcs_note": "duals of the flow-score tree: 44 % of the arcs violate, every tile on the violator "
                               "path; see price_arcs_planted for the kernel's streaming rate",
            "price_arcs_bytes_per_arc": 17, "price_arcs_planted": planted}


# ------------------------------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the device path has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    from smart_crossover import device as dev
    from smart_crossover._native import lib
    from smart_crossover.network_methods.sharded import ShardedDensePricer, row_partition

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    host_group = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
        host_group = dist.new_group(backend="gloo")          # CPU-side waits (no kernel spinning on an idle GPU)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        t = torch.tensor([v], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    if args.score_ctas:
        from smart_crossover._native import lib as _lib
        assert _lib.sx_score_set_tuning(args.score_ctas) == 0
    if args.kruskal_chunk:
        from smart_crossover._native import lib as _lib
        assert _lib.sx_kruskal_set_tuning(args.kruskal_chunk) == 0
    if args.tree_only:
        if args.tree_only == 1:                          # --tree-only 1: the Sinkhorn warm start at 20 000^2
            print(json.dumps(time_sinkhorn(20000, 20000, device)), flush=True)
            return
        if args.tree_only < 0:                           # --tree-only -1: the MCF configuration (1M nodes / 10M arcs)
            print(json.dumps(time_mcf_path(1_000_000, 10_000_000, device, reps=2, cpu=not args.no_cpu)), flush=True)
            return
        T = args.tree_only
        print(json.dumps(time_tree_build(T, T, device, reps=2, cpu=None if args.no_cpu else (min(T, 3000),) * 2,
                                         call_host=True)), flush=True)
        return

    def host_barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(group=host_group)

    ctx = {"world": world, "rank": rank, "device": device, "barrier": barrier, "max_over_ranks": max_over_ranks,
           "host_barrier": host_barrier, "local": local}
    S = D = args.size
    if args.rows:
        S = args.rows
    if args.sweep:
        row0, S_loc = row_partition(S, world, rank)
        P, Q, a = make_points(S, D, device)
        M_loc = make_slab(P, Q, row0, S_loc)
        y_dev = planted_duals(P, Q, a, M_loc, row0, args.violators, world)
        sp = ShardedDensePricer(M_loc, S, row0, args.topk, TOL, variant=args.variant, exchange=args.exchange)
        sweep(args, sp, y_dev, S_loc, D, lib, dev)
        return

    peak, peak_src = measured_peak_gbs()
    steps, warmup = args.steps, max(args.warmup, 3)
    sampler = ClockSampler(local)
    try:
        main_leg = pricing_leg(args, S, D, ctx, steps, warmup, sampler=sampler, want_cpu=not args.no_cpu,
                               want_cold=True)
    finally:
        sampler.stop()                                   # no-op after a normal leg; a failed one leaves no nvidia-smi
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, "", *main_leg["result"])
    main_mgr = manager_leg(args, S, D, ctx, steps, main_leg)
    # second, shorter leg: BASELINE.json configs[3] (dense OT 20 000 x 20 000, "pricing at 1/2/4/8 B200")
    c4_leg, c4_mgr = None, None
    if not args.no_c4 and (S, D) != (args.c4_size, args.c4_size):
        c4_leg = pricing_leg(args, args.c4_size, args.c4_size, ctx, steps, warmup, sampler=None, want_cpu=False,
                             want_cold=False)
        c4_mgr = manager_leg(args, args.c4_size, args.c4_size, ctx, steps, c4_leg)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, "c4_", *c4_leg["result"])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    tree, warm = None, None
    if world == 1 and not args.no_tree:
        torch.cuda.empty_cache()
        cpu = not args.no_cpu
        tree = [time_tree_build(784, 784, device, cpu=(784, 784) if cpu else None),
                time_tree_build(20000, 20000, device, reps=1, cpu=(3000, 3000) if cpu else None, call_host=True),
                time_mcf_path(1_000_000, 10_000_000, device, reps=1, cpu=cpu)]
        warm = time_sinkhorn(20000, 20000, device)

    def roofline_of(leg):
        achieved = 8.0 * leg["S_loc"] * leg["D"] / (leg["kernel_ms"] * 1e-3) / 1e9
        traffic, traffic_src = committed_traffic(leg["S_loc"], leg["D"])
        return {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": peak_src, "kernel": leg["kernel"], "kernel_ms": round(leg["kernel_ms"], 4),
                "kernel_ms_per_rank": leg["kernel_ms_per_rank"], "kernel_ms_source": leg["kernel_ms_source"],
                "algorithmic_bytes_per_arc": 8,
                "frac_of_nominal_8TBs": round(achieved / 8000.0, 4)}

    def workload_of(leg):
        S_, D_ = leg["S"], leg["D"]
        return (f"dense synthetic OT {S_}x{D_} ({S_ * D_:.3g} arcs, {8 * S_ * D_ / 1e9:.1f} GB fp64 cost) "
                f"column-generation pricing pass, row-sharded over {world} GPU(s)")

    L = main_leg
    line = {"metric": METRIC, "value": L["value"], "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": L["ms_per_step"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_of(L),
                       "S": S, "D": D, "topk": args.topk, "tol": TOL, "violating_arcs": L["violating_arcs"],
                       "rows_per_gpu": L["S_loc"], "variant": args.variant, "exchange": L["exchange"],
                       "fused": L["fused"], "row_partition": L["balance"] or "equal shares",
                       "l2": f"inputs larger than L2 ({8 * L['S_loc'] * D / 1e9:.1f} GB per GPU vs 126 MB), no flush needed"},
            "roofline": roofline_of(L), "cpu_baseline": L["cpu_baseline"],
            "e2e": main_mgr if main_mgr is not None else L["e2e"], "e2e_manager_error": L.get("manager_error"),
            "e2e_one_process_per_gpu": L["e2e"], "e2e_pinned": L["e2e_pinned"],
            "topk_digest": L["topk_digest"], "merge_check": L["merge_check"],
            "stage_us_rank0": L["stage_us"], "e2e_cold": L["e2e_cold"], "gpu_launches": L["gpu_launches"],
            "clocks": L["clocks"], "tree_build": tree, "warm_start": warm}
    if c4_leg is not None:
        C = c4_leg
        line["c4"] = {"workload": workload_of(C), "value": C["value"], "unit": UNIT, "ms_per_step": C["ms_per_step"],
                      "steps": steps, "rows_per_gpu": C["S_loc"], "row_partition": C["balance"] or "equal shares",
                      "violating_arcs": C["violating_arcs"],
                      "roofline": roofline_of(C), "stage_us_rank0": C["stage_us"],
                      "e2e": c4_mgr if c4_mgr is not None else C["e2e"], "e2e_one_process_per_gpu": C["e2e"],
                      "e2e_pinned": C["e2e_pinned"], "topk_digest": C["topk_digest"],
                      "merge_check": C["merge_check"], "gpu_launches": C["gpu_launches"]}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def manager_leg(args, S, D, ctx, steps, leg):
    """End to end through the reference's call surface: `OTManager.price(y, K)` /
    `OTManager.check_optimality_condition(x, y)` (net_manager.py:485-497) with a PAGEABLE dual vector, as
    `column_generation` calls it with the LP solver's output (algorithms.py:132).  ONE process: rank 0 drives
    all N GPUs of the job through the manager's persistent pricer (sx_ot_pricer: one worker thread, one
    stream and one fused kernel per GPU); the other ranks of a torchrun job idle on a CPU barrier meanwhile.
    Timed with the host clock around the blocking calls (what the caller sees)."""
    import torch
    world, rank = ctx["world"], ctx["rank"]
    out = None
    ctx["host_barrier"]()
    if rank == 0 and not args.no_manager:
        try:
            from smart_crossover import device as dev
            from smart_crossover.network_methods.net_manager import OTManager
            K = args.topk
            devices = [(ctx["local"] + i) % torch.cuda.device_count() for i in range(world)]
            slabs = dev.CostSlabs(S, D, devices, leg["row_bounds"])
            for g, d in enumerate(devices):
                with torch.cuda.device(d):
                    P, Q, a = make_points(S, D, torch.device("cuda", d))
                    make_slab(P, Q, slabs.row0[g], slabs.rows[g], out=slabs.view(g))
                    del P, Q, a
            slabs.sync()
            mgr = OTManager.from_device_cost(np.full(S, 1.0 / S), np.full(D, 1.0 / D), slabs)
            y = np.array(leg["y_host"], copy=True)               # pageable, as a solver hands it over
            for _ in range(3):
                res = mgr.price(y, K=K)
            t0 = time.perf_counter()
            for _ in range(steps):
                res = mgr.price(y, K=K)
            dt = time.perf_counter() - t0
            assert topk_digest(res.topk_id, res.topk_rc, res.n_violating, res.min_rc) == leg["topk_digest"], \
                "OTManager.price disagrees with the device-timed arm"
            for _ in range(3):
                opt = mgr.check_optimality_condition(None, y)
            t1 = time.perf_counter()
            for _ in range(steps):
                opt = mgr.check_optimality_condition(None, y)
            dt0 = time.perf_counter() - t1
            assert opt == (leg["violating_arcs"] == 0)
            st = mgr._pricer(K).stats()
            G = len(devices)
            blk = 2 * max(K, 1) + 6
            out = {"value": S * D * steps / dt, "unit": UNIT, "ms_per_step": 1e3 * dt / steps,
                   "h2d_bytes_per_step": 8 * (S + G * D), "d2h_bytes_per_step": 8 * blk * G,
                   "call": "OTManager.price(y, K) -- one process drives all GPUs (sx_ot_pricer)",
                   "check_optimality_condition_ms": 1e3 * dt0 / steps,
                   "devices": devices, "fused": st["fused"], "merge_in_kernel": st["merge_in_kernel"],
                   "repeated_passes": st["repeated_passes"], "timer": "host wall clock around the blocking calls",
                   "inputs": "duals y in a pageable NumPy vector every step; each GPU's worker thread stages its "
                             "S_loc + D entries in pinned memory and uploads them; merged result read back; cost "
                             "matrix resident (uploaded / generated once per problem)"}
            mgr._drop_device_state()
            del mgr, slabs
            torch.cuda.empty_cache()
        except AssertionError:                       # a wrong result is never swallowed
            raise
        except Exception as exc:                     # e.g. no peer access between the GPUs of this box: say so and
            out = None                               # let the line fall back to the one-process-per-GPU number
            leg["manager_error"] = f"{type(exc).__name__}: {exc}"
            try:
                torch.cuda.empty_cache()
            except Exception:
                pass
    ctx["host_barrier"]()
    return out


def committed_traffic(S_loc, D):
    """dram read + write bytes of one pricing-kernel launch from the committed ncu captures
    (profiles/price_traffic.json: one entry per captured slab shape).  Exact shape: the captured bytes.  Other
    row counts of the same D (rate-balanced shards, N = 2 / 4): the capture with the nearest row count, its
    traffic / algorithmic ratio applied to this slab's algorithmic bytes -- returned with a note saying so."""
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "price_traffic.json")))
        tj = tj if isinstance(tj, list) else [tj]
        same = [e for e in tj if e["D"] == D]
        for e in same:
            if e["S_loc"] == S_loc:
                return e["traffic_bytes"], "ncu capture of this slab shape (profiles/price_traffic.json)"
        if same:
            e = min(same, key=lambda e: abs(e["S_loc"] - S_loc))
            ratio = e["traffic_bytes"] / e["algorithmic_bytes"]
            return ratio * 8.0 * S_loc * D, (f"scaled: traffic / algorithmic = {ratio:.4f} of the ncu capture at "
                                             f"{e['S_loc']} x {D} applied to {S_loc} x {D}")
    except Exception:
        pass
    return None, None


def topk_digest(ids, rc, count, min_rc):
    """Digest of a pricing result (top-K ids + reduced-cost bits + violator count + min): one value for every
    N proves the row-sharded, exchanged and merged result equals the single-GPU one."""
    h = hashlib.sha256()
    h.update(np.ascontiguousarray(ids, dtype=np.int64).tobytes())
    h.update(np.ascontiguousarray(rc, dtype=np.float64).tobytes())
    h.update(np.int64(count).tobytes())
    h.update(np.float64(min_rc).tobytes())
    return h.hexdigest()[:16]


def pricing_leg(args, S, D, ctx, steps, warmup, sampler, want_cpu, want_cold):
    """Times one dense-OT pricing configuration on the ranks of this job: device-resident arm, stage
    split, N-rank result check, end-to-end arm(s), optional cold upload and CPU baseline."""
    import torch
    import torch.distributed as dist
    from smart_crossover._native import lib
    from smart_crossover.network_methods.sharded import ShardedDensePricer, row_partition
    world, rank, device = ctx["world"], ctx["rank"], ctx["device"]
    barrier, max_over_ranks = ctx["barrier"], ctx["max_over_ranks"]
    K = args.topk
    row0, S_loc = row_partition(S, world, rank)
    P, Q, a = make_points(S, D, device)
    M_loc = make_slab(P, Q, row0, S_loc)
    y_dev = planted_duals(P, Q, a, M_loc, row0, args.violators, world)
    y_host = y_dev.cpu().numpy()
    sp = ShardedDensePricer(M_loc, S, row0, K, TOL, variant=args.variant, exchange=args.exchange,
                            fused=not args.no_fused)
    row_bounds = [S * g // world for g in range(world + 1)]
    balance = None
    if world > 1 and sp.fused and not args.no_balance:
        # Shards sized by measured rate.  An exchanged pass ends when the SLOWEST GPU has delivered its block, and
        # the GPUs of one box stream at rates a few percent apart (power / thermal headroom): time every GPU's own
        # pricing phase (in-kernel stamps: CTA 0's pricing + its wait at the barrier all CTAs reach after pricing)
        # over a few passes of the equal partition, then give each GPU rows in proportion to its rate.
        from smart_crossover.device import balanced_row_bounds
        for _ in range(5):
            sp.enqueue(y_dev)
        ts = []
        for _ in range(8):
            sp.enqueue(y_dev)
            torch.cuda.synchronize()
            ph = sp.pricer.fused_phase_us()
            ts.append(ph["pricing"] + ph["barrier1"])
        spr = torch.zeros(world, dtype=torch.float64, device=device)
        spr[rank] = float(np.median(ts)) / S_loc
        dist.all_reduce(spr, op=dist.ReduceOp.SUM)
        spr = spr.cpu().numpy()
        # time ~ rows only holds when the phase is long against its fixed ramp-up / drain (~6 us) and its
        # run-to-run noise: below 200 us per pass the calibration would mostly redistribute noise
        long_enough = float(np.min(spr * S / world)) >= 200.0
        new_bounds = balanced_row_bounds(S, spr) if long_enough else row_bounds
        balance = {"us_per_1000_rows_equal_partition": [round(float(v) * 1e3, 3) for v in spr],
                   "rows_per_gpu": [new_bounds[g + 1] - new_bounds[g] for g in range(world)],
                   "applied": long_enough}
        if new_bounds != row_bounds:
            del sp, M_loc
            torch.cuda.empty_cache()
            row_bounds = new_bounds
            row0, S_loc = row_bounds[rank], row_bounds[rank + 1] - row_bounds[rank]
            M_loc = make_slab(P, Q, row0, S_loc)
            sp = ShardedDensePricer(M_loc, S, row0, K, TOL, variant=args.variant, exchange=args.exchange,
                                    fused=not args.no_fused)
        barrier()

    # ---- device-resident arm ---------------------------------------------------------------------
    for _ in range(warmup):
        sp.enqueue(y_dev)
    barrier()
    if sampler is not None and rank == 0:
        sampler.start()
    k0 = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    k1 = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    launches0 = sp.launches
    e0.record()
    for i in range(steps):
        out = sp.enqueue(y_dev)
    e1.record()
    launches = sp.launches - launches0                   # kernels of libsxcross inside the timed region only
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    own_ms = e0.elapsed_time(e1)                          # this rank's own clock over the same region
    phases = sp.pricer.fused_phase_us() if sp.fused else None     # in-kernel stamps of the LAST timed pass
    # the result of the last timed step, read before any further pass reuses the pricer's buffers
    count_dev = int(out[3].item())
    assert int(out[6].item()) == 0, "selection status not clean: the timed pass would have to be repeated"
    n_out = int(out[2].item())
    ids_dev, rc_dev = out[1][:n_out].cpu().numpy(), out[0][:n_out].cpu().numpy()
    min_dev = float(lib.sx_key_to_f64(int(out[4].item())))
    # Duration of the pricing kernel.  With the fused pass a step IS one launch of that kernel, so its average
    # launch duration is the timed region / steps (this rank's events around the region).  Only when a step is
    # several launches (separate kernels) are events put around each pricing launch, in a loop of its own: two
    # event records between consecutive kernels cost ~18 us of pipeline bubble (measured), which would otherwise
    # be charged to the step.
    if launches == steps:
        kern_ms, kern_src = own_ms / steps, "timed region / steps (one launch per step)"
    else:
        for i in range(steps):
            sp.enqueue(y_dev, kernel_events=(k0[i], k1[i]))
        barrier()
        kern_ms = float(np.mean([k0[i].elapsed_time(k1[i]) for i in range(steps)]))
        kern_src = "CUDA events around each pricing launch, separate loop"
    digest = topk_digest(ids_dev, rc_dev, count_dev, min_dev)
    value = S * D * steps / (ms_total * 1e-3)

    # ---- N-rank result check: gather every rank's LOCAL top-K block with a plain NCCL all-gather, merge on
    # the host with np.lexsort (independent of sx_exchange_push_ll / the merge kernels) and compare bit for bit
    merge_check = None
    if world > 1:
        local = sp.pricer.block.clone()
        gathered = torch.empty(world, local.numel(), dtype=torch.int64, device=device)
        dist.all_gather_into_tensor(gathered.view(-1), local)
        g = gathered.cpu().numpy()
        Kp = max(K, 1)
        g_rc, g_id = g[:, :Kp].reshape(-1).view(np.float64), g[:, Kp:2 * Kp].reshape(-1)
        real = g_id >= 0
        o = np.lexsort((g_id[real], g_rc[real]))[:K]
        ref_ids, ref_rc = g_id[real][o], g_rc[real][o]
        ref_count = int(g[:, 2 * Kp].sum())
        ref_min = min(float(lib.sx_key_to_f64(int(v))) for v in g[:, 2 * Kp + 1])
        ok = (np.array_equal(ref_ids, ids_dev) and ref_rc.tobytes() == rc_dev.tobytes()
              and ref_count == count_dev and ref_min == min_dev)
        assert ok, f"rank {rank}: exchanged + merged top-K differs from the host merge of the per-rank blocks"
        d_all = [None] * world
        dist.all_gather_object(d_all, digest)
        assert len(set(d_all)) == 1, f"ranks disagree on the merged result: {d_all}"
        merge_check = {"ok": True, "against": "np.lexsort over the NCCL-all-gathered per-rank blocks",
                       "ranks_agree": True, "n_out": n_out}

    # where a step's time goes (separate short loop: the extra events are not in the timed region)
    n_st = 5 if world > 1 else 3
    sev = [[torch.cuda.Event(enable_timing=True) for _ in range(n_st)] for _ in range(20)]
    for i in range(20):
        sp.enqueue(y_dev, stage_events=sev[i])
    torch.cuda.synchronize()
    stage_names = sp.stage_names[:n_st - 1]
    stages = {nm: round(float(np.median([sev[i][q].elapsed_time(sev[i][q + 1]) for i in range(20)])) * 1e3, 1)
              for q, nm in enumerate(stage_names)}
    stages["note"] = "stage times come from a separate loop with CUDA events between the kernels (adds ~18 us per step)"
    if phases is not None:
        stages["fused_kernel_phases_cta0_last_timed_pass"] = phases
    barrier()
    per_rank_kern = [round(kern_ms, 4)]
    if world > 1:                                        # the slowest GPU paces a strong-scaled, exchanged step
        t = torch.zeros(world, dtype=torch.float64, device=device)
        t[rank] = kern_ms
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        per_rank_kern = [round(float(v), 4) for v in t.tolist()]

    # ---- end-to-end arms --------------------------------------------------------------------------------
    # e2e: a PAGEABLE dual vector (what the LP solver returns, algorithms.py:96) in, result out, every step.
    # e2e_pinned: the duals already sit in the pricer's pinned staging buffer (round-1 definition).
    def timed_price(y_arg):
        for _ in range(3):
            r = sp.price(y_arg)
        barrier()
        e0.record()
        for _ in range(steps):
            r = sp.price(y_arg)
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)), r

    y_pageable = np.array(y_host, copy=True)
    e2e_ms, res = timed_price(y_pageable)
    assert res.n_violating == count_dev and topk_digest(res.topk_id, res.topk_rc, res.n_violating, res.min_rc) == digest
    y_pin = sp.y_pinned
    y_pin[:] = y_host
    e2e_pin_ms, res = timed_price(y_pin)
    assert res.n_violating == count_dev
    clocks = sampler.stop() if (sampler is not None and rank == 0) else None

    def e2e_dict(ms, inputs):
        return {"value": S * D * steps / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": sp.h2d_bytes,
                "d2h_bytes_per_step": sp.d2h_bytes, "ms_per_step": ms / steps, "cuda_graph": sp._graph is not None,
                "inputs": inputs}
    e2e = e2e_dict(e2e_ms, "duals y in a pageable NumPy vector every step (copied to pinned staging, this rank's "
                           "S_loc + D entries uploaded), result block read back to the host; cost matrix resident "
                           "(uploaded once per problem, see e2e_cold)")
    e2e_pinned = e2e_dict(e2e_pin_ms, "as e2e, but the duals already sit in the pricer's pinned buffer (y_pinned)")

    # ---- cold end-to-end: also upload this rank's slab of M from pinned host memory (once per problem)
    cold = None
    if want_cold:
        rows_c = min(S_loc, 4000)                       # bounded pinned sample; scaled to the slab
        h_M = torch.empty(rows_c, D, dtype=torch.float64).pin_memory()
        h_M.copy_(M_loc[:rows_c])
        barrier()
        e0.record()
        M_loc[:rows_c].copy_(h_M, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        up_ms = e0.elapsed_time(e1) * (S_loc / rows_c)
        cold = {"value": S * D / ((max_over_ranks(up_ms) + e2e_ms / steps) * 1e-3), "unit": UNIT,
                "h2d_bytes": 8 * S_loc * D, "note": f"upload time scaled from a {rows_c}-row pinned sample"}
        del h_M

    cpu_baseline = None
    if want_cpu and rank == 0:
        rows_h = min(S_loc, 16384)                       # ~5e8-1e9 arcs: a few seconds of single-core NumPy per repetition
        M_h = M_loc[:rows_h].cpu().numpy()
        y_h = np.concatenate([y_host[row0:row0 + rows_h], y_host[S:]])
        rate, dt = cpu_price_rate(M_h, y_h, K, 1, 2)
        cpu_baseline = {"value": rate, "unit": UNIT, "cores": 1, "kind": "port",
                        "sample": f"first {rows_h} of {S} rows x {D} cols ({M_h.size:.3g} arcs), best of 2, "
                                  f"oracle NumPy restatement of net_manager.py:474-497, host has {os.cpu_count()} cpus"}
        del M_h

    leg = {"S": S, "D": D, "S_loc": S_loc, "value": value, "ms_per_step": ms_total / steps, "kernel_ms": kern_ms,
           "kernel_ms_per_rank": per_rank_kern, "kernel": sp.pricing_kernel_name, "kernel_ms_source": kern_src,
           "stage_us": stages,
           "gpu_launches": launches, "violating_arcs": count_dev, "topk_digest": digest, "merge_check": merge_check,
           "e2e": e2e, "e2e_pinned": e2e_pinned, "e2e_cold": cold, "cpu_baseline": cpu_baseline, "clocks": clocks,
           "exchange": sp.exchange, "fused": sp.fused, "y_host": y_host, "row_bounds": row_bounds, "balance": balance,
           "result": (count_dev, min_dev, ids_dev, rc_dev)}
    del sp, M_loc, y_dev
    torch.cuda.empty_cache()
    barrier()
    return leg


def sweep(args, sp, y_dev, S_loc, D, lib, dev):
    """Pricing-kernel variants and tunings, kernel-only GB/s (CUDA events, 20 reps after 3 warm-ups)."""
    import torch
    if args.sweep_ab:
        # entries: shape index, or shape:l2promo:evict (TMA options)
        idx = [t for t in args.sweep_ab.split(",")]
        ms = {i: [] for i in idx}
        sp.variant = 0
        for rnd in range(8):
            for i in idx:
                parts = [int(v) for v in i.split(":")]
                lib.sx_price_set_tuning(parts[0], 0)
                lib.sx_price_set_tma_options(parts[1] if len(parts) > 1 else 3, parts[2] if len(parts) > 2 else 1)
                for _ in range(2):
                    sp.enqueue(y_dev)
                k0 = [torch.cuda.Event(enable_timing=True) for _ in range(10)]
                k1 = [torch.cuda.Event(enable_timing=True) for _ in range(10)]
                for r in range(10):
                    sp.enqueue(y_dev, kernel_events=(k0[r], k1[r]))
                torch.cuda.synchronize()
                ms[i] += [k0[r].elapsed_time(k1[r]) for r in range(10)]
        for i in idx:
            print(json.dumps({"tma_shape": i, "kernel_ms_median": round(float(np.median(ms[i])), 4),
                              "kernel_ms_min": round(float(min(ms[i])), 4),
                              "GBs_median": round(8.0 * S_loc * D / (np.median(ms[i]) * 1e-3) / 1e9, 1)}), flush=True)
        lib.sx_price_set_tuning(6, 16)
        lib.sx_price_set_tma_options(3, 1)
        return
    res = []
    shapes = ["16x6 8w", "16x6 16w", "32x3 8w", "32x3 16w", "16x7 16w", "8x12 16w", "16x3 8w x2cta", "8x6 8w x2cta",
              "24x4 16w", "20x5 16w", "12x9 16w", "12x4 8w x2cta", "8x7 8w x2cta", "8x4 8w x3cta"]
    confs = [(f"tma {nm}", 0, (i, 0)) for i, nm in enumerate(shapes)]
    confs += [("vec", 1, (-1, 4)), ("vec", 1, (-1, 8)), ("vec", 1, (-1, 16)), ("scalar", 2, (-1, 8)),
              ("scalar", 2, (-1, 16))]
    for name, variant, tune in confs:
        lib.sx_price_set_tuning(*tune)
        sp.variant = variant
        for _ in range(3):
            sp.enqueue(y_dev)
        torch.cuda.synchronize()
        k0 = [torch.cuda.Event(enable_timing=True) for _ in range(20)]
        k1 = [torch.cuda.Event(enable_timing=True) for _ in range(20)]
        for i in range(20):
            sp.enqueue(y_dev, kernel_events=(k0[i], k1[i]))
        torch.cuda.synchronize()
        ms = [k0[i].elapsed_time(k1[i]) for i in range(20)]
        gbs = 8.0 * S_loc * D / (np.median(ms) * 1e-3) / 1e9
        res.append({"variant": name, "tuning": tune, "kernel_ms_median": round(float(np.median(ms)), 4),
                    "kernel_ms_min": round(float(min(ms)), 4), "GBs": round(gbs, 1)})
        print(json.dumps(res[-1]), flush=True)
    lib.sx_price_set_tuning(6, 16)


if __name__ == "__main__":
    main()

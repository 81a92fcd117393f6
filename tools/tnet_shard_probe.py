"""TNET crossover inputs on a row-sharded, device-resident OT problem: the flow scored on every shard's GPU, the
head of the Kruskal order selected across the shards (`sx_order_head_sharded_h`), Kruskal on the first GPU, the
tree flows and push, and the queue slices of a column-generation schedule -- against the single-GPU host route
(`get_sorted_flows` + `tree_basis_identify` on host arrays) at the smaller size.

Workload: bench.py's squared-Euclidean costs generated slab by slab on the device (no host copy), seeded marginals,
and as the flow the sharded Sinkhorn plan (`warm_start.sinkhorn(..., as_slabs=True)`) after a FIXED number of
iterations (--sinkhorn-iters, stopThr = 0), reg = 0.01 * median of the first 64 cost rows.

For G shards: shard g on visible device g mod (device count).  With fewer GPUs than shards, shards share a GPU and
run one after the other (the emulation the tests use): G > 1 then measures the extra launches and round trips of
the sharded selection, not a multi-GPU speed-up.

Times are host clocks around calls that end in a device synchronise (the library's sharded entry is blocking),
median of --reps after one warm-up.  Per-shard scoring times come from CUDA events around each shard's kernel.

    python tools/tnet_shard_probe.py --sizes 20000 60000 --shards 1 2 4 8 --out profiles/r03_tnet_shard_probe.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "smart-crossover_b200"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from smart_crossover import device as dev  # noqa: E402
from smart_crossover.formats import OptTransport  # noqa: E402
from smart_crossover.network_methods.net_manager import DeviceResidentCost, OTManager  # noqa: E402
from smart_crossover.network_methods.tree_BI import PREFIX_FACTOR, _device_tree, push_tree_to_bfs  # noqa: E402
from smart_crossover.warm_start import sinkhorn  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return [line.strip() for line in q.stdout.strip().splitlines()]


def sync_all():
    for i in range(torch.cuda.device_count()):
        torch.cuda.synchronize(i)


def timed(fn, reps):
    """(median seconds, last result) of `reps` calls after one warm-up call."""
    fn()
    ts, r = [], None
    for _ in range(reps):
        sync_all()
        t0 = time.perf_counter()
        r = fn()
        sync_all()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), r


def score_ms_per_shard(flow, s, d):
    """CUDA-event time of each shard's sx_score_ot (ms)."""
    out = []
    for g, dv in enumerate(flow.devices):
        with torch.cuda.device(dv):
            r0 = flow.row0[g]
            s_g = torch.from_numpy(np.ascontiguousarray(s[r0:r0 + flow.rows[g]])).cuda()
            d_g = torch.from_numpy(np.ascontiguousarray(d)).cuda()
            dst = torch.empty(flow.rows[g] * flow.D, dtype=torch.float64, device="cuda")
            dev.score_ot(flow.t[g], s_g, d_g, want_hist=True, out=dst)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            dev.score_ot(flow.t[g], s_g, d_g, want_hist=True, out=dst)
            e1.record()
            e1.synchronize()
            out.append(round(e0.elapsed_time(e1), 3))
            del dst
    return out


def cg_slices(m, n, rounds):
    left, target = 0, int(10 * m) if n / m > 1000 else int(1.2 * m)
    for _ in range(rounds):
        if left >= n:
            break
        right = min(target, n)
        yield left, right
        left, target = right, 2 * target


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[20000, 60000])
    ap.add_argument("--shards", type=int, nargs="+", default=[1, 2, 4, 8])
    ap.add_argument("--sinkhorn-iters", type=int, default=30)
    ap.add_argument("--cg-rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--host-route-max", type=int, default=20000, help="largest size that also runs the host route")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    n_vis = torch.cuda.device_count()
    d0 = torch.device("cuda", 0)
    torch.cuda.set_device(d0)
    out = {"cards": card(), "visible_gpus": n_vis, "torch": torch.__version__, "flow": "sharded Sinkhorn plan, "
           f"{args.sinkhorn_iters} iterations, stopThr = 0", "sizes": []}
    for n_side in args.sizes:
        S = D = n_side
        N, n = S + D, S * D
        P, Q, _ = bench.make_points(S, D, d0, seed=20260004)
        g_ = torch.Generator(device=d0).manual_seed(5)
        s = (torch.rand(S, generator=g_, device=d0, dtype=torch.float64) + 0.1)
        dd = (torch.rand(D, generator=g_, device=d0, dtype=torch.float64) + 0.1)
        s, dd = (s / s.sum()).cpu().numpy(), (dd / dd.sum()).cpu().numpy()
        reg = 0.01 * float(bench.make_slab(P, Q, 0, 64).median().item())
        rec = {"S": S, "D": D, "reg": reg, "shards": []}
        ref_tree = None
        for G in args.shards:
            devices = [i % n_vis for i in range(G)]
            slabs = dev.CostSlabs(S, D, devices)
            for g, dv in enumerate(devices):
                bench.make_slab(P.to(torch.device("cuda", dv)), Q.to(torch.device("cuda", dv)), slabs.row0[g],
                                slabs.rows[g], out=slabs.view(g))
            slabs.sync()
            flow = sinkhorn(s, dd, slabs, reg, numItermax=args.sinkhorn_iters, stopThr=0.0, as_slabs=True)
            ot = OptTransport(s, dd, DeviceResidentCost(slabs))
            mgr = OTManager(ot)
            r = {"G": G, "devices": devices, "shards_share_a_gpu": len(set(devices)) < G}
            r["score_ms_per_shard_events"] = score_ms_per_shard(flow, s, dd)
            t, (queue, scores) = timed(lambda: mgr.get_sorted_flows(flow), args.reps)
            r["get_sorted_flows_ms"] = round(t * 1e3, 2)
            T = PREFIX_FACTOR * N
            t, head = timed(lambda: dev.order_head_sharded(scores.slabs, T, hists=scores.hists), args.reps)
            r["head_kruskal_T"] = T
            r["head_kruskal_ms_incl_gather"] = round(t * 1e3, 2)
            r["head_kruskal_arcs"] = None if head is None else int(head.numel())
            with torch.cuda.device(devices[0]):
                t, (tree_t, n_t) = timed(lambda: dev.kruskal(head, N, S=S, D=D), args.reps)
            r["kruskal_ms"] = round(t * 1e3, 2)
            r["kruskal_complete"] = int(n_t.item()) == N - 1
            tree_t, nt = _device_tree(ot, scores, mgr._sorted)
            tree = tree_t[:nt].cpu().numpy()
            t, (_, push_iter) = timed(lambda: push_tree_to_bfs(mgr, tree), args.reps)
            r["tree_flows_plus_push_ms"] = round(t * 1e3, 2)
            r["push_iter"] = push_iter
            mats = []
            for a, b in cg_slices(N, n, args.cg_rounds):
                before = queue._head.size
                sync_all()
                t0 = time.perf_counter()
                queue[a:b]
                sync_all()
                if queue._head.size != before:
                    mats.append({"slice": [a, b], "materialised": int(queue._head.size),
                                 "ms": round((time.perf_counter() - t0) * 1e3, 2)})
            r["queue_materialisations"] = mats
            if ref_tree is None:
                ref_tree = tree
            r["tree_equals_G1"] = bool(np.array_equal(tree, ref_tree))
            if G == args.shards[0] and n_side <= args.host_route_max:
                # single-GPU host route on the same flow: host x -> get_sorted_flows (full sort, n-sized downloads)
                # -> tree_basis_identify; compared arc for arc
                x_h = np.concatenate([dev.to_host(t_) for t_ in flow.t]).ravel()
                M_h = np.concatenate([dev.to_host(slabs.view(g).contiguous()) for g in range(G)])
                host = OTManager(OptTransport(s, dd, M_h))
                t_sf, (hq, hs) = timed(lambda: host.get_sorted_flows(x_h), args.reps)
                t_tb, _ = timed(lambda: _device_tree(host.ot, hs, host._sorted), args.reps)
                htree, hnt = _device_tree(host.ot, hs, host._sorted)
                r["host_route"] = {"get_sorted_flows_ms": round(t_sf * 1e3, 2), "device_tree_ms": round(t_tb * 1e3, 2),
                                   "tree_equal_arc_for_arc": bool(np.array_equal(htree[:hnt].cpu().numpy(), tree))}
                del x_h, M_h, host, hq, hs
            rec["shards"].append(r)
            print(json.dumps({"size": n_side, **r}), flush=True)
            del flow, slabs, mgr, queue, scores, head, ot
            torch.cuda.empty_cache()
        out["sizes"].append(rec)
    out["cards_after"] = card()
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()

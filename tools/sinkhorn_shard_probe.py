"""Sinkhorn warm start over row-sharded cost slabs (`sx_sinkhorn_ot_sharded_h`) against the single-GPU call
(`sx_sinkhorn_ot`) on the same seeded problem: bench.py's device-generated squared-Euclidean costs, seeded
marginals, reg = 0.01 * median of the first 64 rows (as bench's `time_sinkhorn`), stopThr = 0.

For N ranks: shard g on visible device g mod (device count); with fewer GPUs than ranks, several ranks share a
GPU and run one after the other on its stream (the emulation the tests use), so N > 1 then measures what the
push / fold exchange and the extra launches cost, not a multi-GPU speed-up.

Per-iteration times are host-clock differences between the medians of 5 blocking calls of n_lo and of n_hi
iterations (after a warm-up call): the per-call set-up (allocation, uploads, read-back) cancels out and is reported
separately.
  - fp64-equivalent GB/s per device: 16 B per arc and iteration over the devices in use;
  - efficiency against N = 1: (t_1 / t_N) / devices in use;
  - host enqueue per iteration, measured directly: the kernel-launch calls torch.profiler records on the host
    during one call of 12 iterations at the measured size (stopThr = 0: nothing synchronises inside the loop, and
    12 iterations do not fill a stream's launch queue): the span from the loop's first to its last launch, and
    the time spent inside the launch calls, each per iteration (under the profiler, which adds its own cost
    per call);
  - launch-bound iteration: the same call at S = 128 N, D = 256, where every kernel takes a few microseconds: the
    larger of the host enqueue and the chain of 4 N launches on the GPU (one GPU when ranks share it);
  - max relative difference of f, g and the plan against the N = 1 result;
  - same-run comparison: sx_sinkhorn_ot and the N = 1 sharded call, alternated.

    python tools/sinkhorn_shard_probe.py --sizes 20000 60000 --ranks 1 2 4 8 --out sinkhorn_probe.json
"""
import argparse
import ctypes
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
from smart_crossover._native import check, lib  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return [line.strip() for line in q.stdout.strip().splitlines()]


def make_slabs(P, Q, S, D, devices):
    sl = dev.CostSlabs(S, D, devices)
    for g, d in enumerate(devices):
        bench.make_slab(P.to(torch.device("cuda", d)), Q.to(torch.device("cuda", d)), sl.row0[g], sl.rows[g],
                        out=sl.view(g))
    sl.sync()
    return sl


def sharded(sl, a, b, reg, iters, x_out=None):
    """One blocking call; returns (seconds, f, g, iterations)."""
    G, S, D = len(sl.devices), sl.S, sl.D
    f, g = np.empty(S), np.empty(D)
    it, err = ctypes.c_int64(0), ctypes.c_double(0.0)
    xs = (ctypes.c_void_p * G)(*[x.data_ptr() for x in x_out]) if x_out is not None else None
    t0 = time.perf_counter()
    check(lib.sx_sinkhorn_ot_sharded_h(G, (ctypes.c_int * G)(*sl.devices),
                                       (ctypes.c_void_p * G)(*[t.data_ptr() for t in sl.t]),
                                       (ctypes.c_int64 * (G + 1))(*sl.row_bounds), sl.ld, S, D, a.ctypes.data,
                                       b.ctypes.data, reg, iters, 0.0, 10, f.ctypes.data, g.ctypes.data, xs,
                                       ctypes.byref(it), ctypes.byref(err)), "sx_sinkhorn_ot_sharded_h")
    return time.perf_counter() - t0, f, g, it.value


def per_iter(run, n_lo, n_hi, reps=5):
    """(ms per iteration, ms of fixed per-call cost) from the medians of blocking calls of n_lo / n_hi iterations."""
    run(2)
    lo = np.median([run(n_lo) for _ in range(reps)])
    hi = np.median([run(n_hi) for _ in range(reps)])
    ms = (hi - lo) / (n_hi - n_lo) * 1e3
    return ms, lo * 1e3 - n_lo * ms


def enqueue_us(sl, a, b, reg, iters=12):
    """Host enqueue per iteration (us): span of the loop's launch calls and time inside them, from torch.profiler's
    host-side record of one call; None when the profiler recorded fewer launches than the loop makes."""
    from torch.profiler import ProfilerActivity, profile
    G = len(sl.devices)
    sharded(sl, a, b, reg, 2)
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        sharded(sl, a, b, reg, iters)
    names = sorted({e.name for e in prof.events() if "LaunchKernel" in e.name})
    name = next((n for n in names if n.startswith("cudaLaunchKernel")), names[0] if names else None)
    ev = sorted((e for e in prof.events() if e.name == name), key=lambda e: e.time_range.start)
    loop = ev[3 * G:]                                   # the set-up launches 3 kernels per rank before the loop
    out = {"api": name, "launches_seen": len(ev), "launches_expected": 3 * G + 4 * G * iters,
           "span_us_per_iter": None, "in_launch_calls_us_per_iter": None}
    if len(loop) == 4 * G * iters:
        out["span_us_per_iter"] = round((loop[-1].time_range.end - loop[0].time_range.start) / iters, 2)
        out["in_launch_calls_us_per_iter"] = round(
            sum(e.time_range.end - e.time_range.start for e in loop) / iters, 2)
    return out


def rel_diff(x, ref):
    """max |x - ref| / max |ref| (potentials cross zero)"""
    return float(np.max(np.abs(x - ref)) / np.max(np.abs(ref)))


def plan_diff(X, X1, sl):
    """max |X - X1| / |X1| over every shard (entries that underflow to 0 count against 1e-300), on the device,
    2000 rows at a time."""
    worst = 0.0
    for g in range(len(sl.devices)):
        r0 = sl.row0[g]
        for r in range(0, sl.rows[g], 2000):
            e = min(sl.rows[g], r + 2000)
            ref = X1[r0 + r:r0 + e]
            x = X[g][r:e].to(ref.device)
            worst = max(worst, float(((x - ref).abs() / ref.abs().clamp_min(1e-300)).max().item()))
    return worst


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[20000, 60000])
    ap.add_argument("--ranks", type=int, nargs="+", default=[1, 2, 4, 8])
    ap.add_argument("--iters", type=int, nargs=2, default=None, help="n_lo n_hi (default: by size)")
    ap.add_argument("--alternate", type=int, default=4, help="rounds of the same-run comparison")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    n_vis = torch.cuda.device_count()
    d0 = torch.device("cuda", 0)
    torch.cuda.set_device(d0)
    out = {"cards": card(), "visible_gpus": n_vis, "torch": torch.__version__, "sizes": []}
    for n in args.sizes:
        S = D = n
        n_lo, n_hi = args.iters or ((10, 410) if n <= 20000 else (4, 64))      # windows of 0.6-0.9 s
        P, Q, _ = bench.make_points(S, D, d0, seed=20260004)
        g_ = torch.Generator(device=d0).manual_seed(5)
        a = torch.rand(S, generator=g_, device=d0, dtype=torch.float64) + 0.1
        b = torch.rand(D, generator=g_, device=d0, dtype=torch.float64) + 0.1
        a /= a.sum(); b /= b.sum()
        a_h, b_h = a.cpu().numpy(), b.cpu().numpy()
        reg = 0.01 * float(bench.make_slab(P, Q, 0, 64).median().item())
        rec = {"S": S, "D": D, "reg": reg, "iters_lo_hi": [n_lo, n_hi], "ranks": []}
        ref = None
        for N in args.ranks:
            devices = [i % n_vis for i in range(N)]
            sl = make_slabs(P, Q, S, D, devices)
            ms, fixed_ms = per_iter(lambda k: sharded(sl, a_h, b_h, reg, k)[0], n_lo, n_hi)
            X = [torch.empty(sl.rows[g], D, dtype=torch.float64, device=sl.t[g].device) for g in range(N)]
            _, f, g, _ = sharded(sl, a_h, b_h, reg, n_hi, X)
            n_dev = len(set(devices))
            r = {"N": N, "devices": devices, "ranks_share_a_gpu": n_dev < N, "ms_per_iter": round(ms, 4),
                 "per_call_fixed_ms": round(fixed_ms, 2),
                 "fp64_equiv_GBps_per_device": round(16.0 * S * D / (ms * 1e-3) / 1e9 / n_dev, 1)}
            r["host_enqueue"] = enqueue_us(sl, a_h, b_h, reg)
            # launch-bound iteration: tiny shards, same devices
            tiny = dev.CostSlabs(128 * N, 256, devices)
            for t in tiny.t:
                t.fill_(1.0)
            tiny.sync()
            ta, tb = np.full(128 * N, 1.0 / (128 * N)), np.full(256, 1.0 / 256)
            r["launch_bound_us_per_iter"] = round(
                per_iter(lambda k: sharded(tiny, ta, tb, 0.1, k)[0], 200, 1200)[0] * 1e3, 2)
            del tiny
            if ref is None:
                ref = (ms, f, g, torch.cat([x.to(d0) for x in X]) if N > 1 else X[0])
                r["efficiency_vs_N1"] = 1.0
            else:
                r["efficiency_vs_N1"] = round(ref[0] / ms / n_dev, 3)
                r["max_rel_diff_vs_N1"] = {"f": rel_diff(f, ref[1]), "g": rel_diff(g, ref[2]),
                                           "plan": plan_diff(X, ref[3], sl)}
            if N == 1:
                # same-run comparison with the single-GPU entry on the same matrix (slab 0 is the whole matrix)
                M = sl.t[0][:, :D]
                fd = torch.empty(S, dtype=torch.float64, device=d0)
                gd = torch.empty(D, dtype=torch.float64, device=d0)
                ws = dev._ws(lib.sx_sinkhorn_workspace_bytes(S, D), d0)
                it_h, err_h = ctypes.c_int64(0), ctypes.c_double(0.0)

                def single(k):
                    t0 = time.perf_counter()
                    check(lib.sx_sinkhorn_ot(dev._ptr(M), sl.ld, S, D, dev._ptr(a), dev._ptr(b), reg, k, 0.0, 10,
                                             dev._ptr(fd), dev._ptr(gd), None, ctypes.byref(it_h),
                                             ctypes.byref(err_h), dev._ptr(ws), ws.numel(), dev._stream()),
                          "sx_sinkhorn_ot")
                    torch.cuda.synchronize()
                    return time.perf_counter() - t0
                alt = {"sx_sinkhorn_ot": [], "sharded_N1": []}
                for _ in range(args.alternate):
                    alt["sx_sinkhorn_ot"].append(round(per_iter(single, n_lo, n_hi)[0], 4))
                    alt["sharded_N1"].append(round(per_iter(lambda k: sharded(sl, a_h, b_h, reg, k)[0],
                                                            n_lo, n_hi)[0], 4))
                single(n_hi)
                torch.cuda.synchronize()
                alt["f_g_bitwise_equal"] = bool(np.array_equal(fd.cpu().numpy().view(np.int64), f.view(np.int64))
                                                and np.array_equal(gd.cpu().numpy().view(np.int64),
                                                                   g.view(np.int64)))
                alt["median_ms_per_iter"] = {k: float(np.median(v)) for k, v in alt.items() if isinstance(v, list)}
                r["same_run_comparison"] = alt
                del ws, fd, gd
            rec["ranks"].append(r)
            print(json.dumps({"size": n, **r}), flush=True)
            del X, sl
            torch.cuda.empty_cache()
        out["sizes"].append(rec)
        del ref
        torch.cuda.empty_cache()
    out["cards_after"] = card()
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()

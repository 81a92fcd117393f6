"""What pricing the big-M border next to the base slabs costs: a pass of the bordered pricer
(`sx_ot_pricer_create_bigm`, the extension of cnet_ot on a device-resident problem) against a pass of the plain
pricer over the same S x D slabs (`sx_ot_pricer_create`), alternated in one run.

Costs are bench.py's device-generated squared-Euclidean ones, bigM = (S + D) * max(M) as `network_crossover` sets
it.  Duals are planted: y0 = (a, b), b_j = min_i (M_ij + a_i), every inner reduced cost >= 0; then 0.1 % of the
columns are raised by 2e-6 (inner violators), u_S and v_D are set so that about 0.1 % of the artificial row and of
the artificial column violate.  The plain pricer gets the same inner duals.  Times are host clocks around the
blocking `price` calls (median, 10-90 % range), after warm-up passes.  Shard g on device g; a rank count above
the visible GPU count is skipped.

    python tools/cnet_bigm_probe.py --sizes 20000 60000 --ranks 1 2 4 8 --out profiles/r03_cnet_bigm_probe.json
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


def duals(sl, seed):
    """Host (y_src of S + 1, y_dst of D + 1) for the extension, and bigM."""
    rng = np.random.default_rng(seed)
    S, D = sl.S, sl.D
    a = rng.random(S)
    b = np.full(D, np.inf)
    for g, d in enumerate(sl.devices):
        r0 = sl.row0[g]
        a_g = torch.from_numpy(a[r0:r0 + sl.rows[g]]).to(torch.device("cuda", d))
        b = np.minimum(b, torch.amin(sl.view(g) + a_g[:, None], dim=0).cpu().numpy())
    b[rng.random(D) < 1e-3] += 2e-6
    bigM = (S + D) * sl.max()
    v_D = bigM + np.quantile(a, 1e-3)                   # rc(i, D) = bigM - (v_D - u_i) < 0 for ~0.1 % of the rows
    u_S = np.quantile(b, 1 - 1e-3) - bigM               # rc(S, j) = bigM - (v_j - u_S) < 0 for ~0.1 % of the columns
    return np.append(a, u_S), np.append(b, v_D), float(bigM)


def stats(ts):
    ts = np.asarray(ts) * 1e3
    return {"median_ms": round(float(np.median(ts)), 4), "p10_ms": round(float(np.percentile(ts, 10)), 4),
            "p90_ms": round(float(np.percentile(ts, 90)), 4), "n": int(ts.size)}


def run(S, D, G, K, reps, warm):
    devices = list(range(G))
    gen = torch.Generator().manual_seed(S + D)
    P, Q = torch.rand(S, 2, generator=gen, dtype=torch.float64), torch.rand(D, 2, generator=gen, dtype=torch.float64)
    sl = make_slabs(P, Q, S, D, devices)
    y_src, y_dst, bigM = duals(sl, S)
    plain = dev.OTPricer(sl, K)
    bord = dev.OTPricer(sl, K, bigm=(bigM, 0.0))
    t_plain, t_bord = [], []
    for it in range(warm + reps):
        for pr, ys, yd, acc in ((plain, y_src[:S], y_dst[:D], t_plain), (bord, y_src, y_dst, t_bord)):
            t0 = time.perf_counter()
            pr.price(ys, yd)
            dt = time.perf_counter() - t0
            if it >= warm:
                acc.append(dt)
        if it == 0:
            r_plain, r_bord = plain.price(y_src[:S], y_dst[:D]), bord.price(y_src, y_dst)
    out = {"S": S, "D": D, "ranks": G, "devices": devices, "K": K, "bigM": bigM,
           "violators_plain": r_plain.n_violating, "violators_bordered": r_bord.n_violating,
           "border_violators": r_bord.n_violating - r_plain.n_violating,
           "plain": stats(t_plain), "bordered": stats(t_bord),
           "stats_bordered": bord.stats()}
    out["extra_ms_median"] = round(out["bordered"]["median_ms"] - out["plain"]["median_ms"], 4)
    plain.close()
    bord.close()
    del sl
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[20000, 60000])
    ap.add_argument("--ranks", type=int, nargs="+", default=[1, 2, 4, 8])
    ap.add_argument("--K", type=int, nargs="+", default=[0, 64])
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warm", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_cnet_bigm_probe.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("the probe needs CUDA devices")
    n_vis = torch.cuda.device_count()
    rec = {"card": card(), "visible_gpus": n_vis, "torch": torch.__version__, "runs": []}
    for n in args.sizes:
        for G in args.ranks:
            if G > n_vis:
                rec["runs"].append({"S": n, "D": n, "ranks": G, "skipped": f"{n_vis} GPU(s) visible"})
                continue
            for K in args.K:
                r = run(n, n, G, K, args.reps, args.warm)
                print(json.dumps(r), flush=True)
                rec["runs"].append(r)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()

"""Both walks of the fused pricing pass on one GPU: the fp64 walk (streams M, 8 B per arc) and the lower-bound
walk (streams the 4-byte copy of sx_cost_lb_build, and re-reads the exact cost of every flagged arc).

For each walk: kernel time from CUDA events around a loop of launches, bytes moved (the stream, plus one 32 B
sector per flagged arc's sector for the lower-bound walk, plus the candidate writes), the achieved GB/s and
CTA 0's in-kernel phase stamps of the last pass.  The inputs are bench.py's (seeded points, planted duals).

    python tools/lb_probe.py --size 60000 --violators 1e-4 --launches 100
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "smart-crossover_b200"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from smart_crossover import device as dev  # noqa: E402


def flagged_sectors(M, lb, y, S, D, tol):
    """Arcs whose lower-bound reduced cost is below -tol (or NaN) and the 32 B sectors of M they fall in (what
    the walk re-reads once the running minimum is below -tol, i.e. after the first violator)."""
    v = y[S:S + D]
    n_arcs = n_sect = 0
    pad = (-D) % 4
    for r in range(0, S, 2000):
        e = min(S, r + 2000)
        L = (lb[r:e, :D].to(torch.int64) << 32).view(torch.float64)
        rc_lb = L - (v[None, :] - y[r:e, None])
        f = ~(rc_lb >= -tol)
        n_arcs += int(f.sum().item())
        if pad:
            f = torch.nn.functional.pad(f, (0, pad))
        n_sect += int(f.view(e - r, -1, 4).any(dim=2).sum().item())
    return n_arcs, n_sect


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=60000)
    ap.add_argument("--violators", type=float, default=1e-4)
    ap.add_argument("--topk", type=int, default=1024)
    ap.add_argument("--launches", type=int, default=100)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    S = D = args.size
    device = torch.device("cuda", 0)
    torch.cuda.set_device(device)
    P, Q, a = bench.make_points(S, D, device)
    M = bench.make_slab(P, Q, 0, S)
    y = bench.planted_duals(P, Q, a, M, 0, args.violators, 1)
    lb = dev.cost_lb(M)
    torch.cuda.synchronize()
    n_flag, n_sect = flagged_sectors(M, lb, y, S, D, bench.TOL)
    props = torch.cuda.get_device_properties(device)
    out = {"gpu": props.name, "S": S, "D": D, "K": args.topk, "violators_target": args.violators,
           "flagged_arcs": n_flag, "flagged_sectors": n_sect, "launches": args.launches, "walks": {}}
    digests = {}
    for name, use_lb in (("fp64", False), ("lower_bound", True)):
        pr = dev.Pricer(device, args.topk, fused=True)
        call = lambda: pr.price_dense_fused(M, M.stride(0), 0, S, D, y[:S], y[S:], bench.TOL,
                                            lb=lb if use_lb else None)
        for _ in range(5):
            call()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.launches):
            call()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.launches
        res = pr.fetch()
        digests[name] = bench.topk_digest(res.topk_id, res.topk_rc, res.n_violating, res.min_rc)
        cand = pr.n_candidates()
        stream = (4 if use_lb else 8) * S * D
        moved = stream + (32 * n_sect if use_lb else 0) + 16 * cand
        out["walks"][name] = {"kernel_ms": round(ms, 4), "walk_reported": pr.fused_walk(),
                              "bytes_moved": moved, "bytes_stream": stream, "candidates": cand,
                              "achieved_GBps": round(moved / (ms * 1e-3) / 1e9, 1),
                              "fp64_equivalent_GBps": round(8 * S * D / (ms * 1e-3) / 1e9, 1),
                              "n_violating": res.n_violating, "cta0_phases_us": pr.fused_phase_us()}
    assert digests["fp64"] == digests["lower_bound"], digests
    out["topk_digest"] = digests["fp64"]
    out["speedup"] = round(out["walks"]["fp64"]["kernel_ms"] / out["walks"]["lower_bound"]["kernel_ms"], 3)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

"""bench.py --dump-outputs: the result of the last timed step, as a caller of the timed path receives it, written as
float64 .npy files that two runs with the same arguments reproduce."""
import itertools
import json
import os
import subprocess
import sys
import types

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")
NAMES = ("n_violating", "min_rc", "topk_id", "topk_rc")


def _run(cwd, *args):
    out = subprocess.run([sys.executable, BENCH, *args], cwd=cwd, check=True, capture_output=True, text=True).stdout
    return json.loads(out.strip().splitlines()[-1])


def _load(d, prefix=""):
    return {n: np.load(os.path.join(d, prefix + n + ".npy")) for n in NAMES}


def test_reference_arm_dump_does_not_depend_on_host_speed_and_runs_steps_passes(tmp_path, monkeypatch, capsys):
    """Two runs whose clocks make the host look a million times faster or slower (which would size the row sample
    at S or at its floor) dump the same result, and each prices exactly warmup + steps times.  S = 2000 is larger
    than the dump's 512-row sample, so a clamp to S cannot hide a timed size."""
    import bench
    from oracle import network_oracle as orc
    real, calls = orc.price_dense_ot_blocked, []
    monkeypatch.setattr(orc, "price_dense_ot_blocked", lambda *a, **kw: calls.append(1) or real(*a, **kw))
    runs = []
    for steps, warmup, tick in ((2, 1, 1e-6), (3, 0, 1e3)):
        clock = itertools.count(0.0, tick)
        monkeypatch.setattr(bench, "time", types.SimpleNamespace(perf_counter=lambda c=clock: next(c)))
        d = tmp_path / f"s{steps}"
        monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--size", "2000", "--topk", "64",
                                          "--steps", str(steps), "--warmup", str(warmup), "--dump-outputs", str(d)])
        calls.clear()
        bench.run_reference(bench.parse())
        line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
        assert len(calls) == warmup + steps and line["steps"] == steps
        assert line["config"]["rows_per_step"] == 512
        runs.append(_load(d))
    a, b = runs
    for n in NAMES:
        assert a[n].dtype == np.float64 and a[n].tobytes() == b[n].tobytes(), n
    k = a["topk_id"].size
    assert k == min(64, int(a["n_violating"][0])) and k == a["topk_rc"].size and np.unique(a["topk_id"]).size == k
    assert a["topk_rc"][0] == a["min_rc"][0] and np.all(np.diff(a["topk_rc"]) >= 0) and np.all(a["topk_rc"] < -1e-6)


def test_dump_outputs_samples_a_long_topk(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_MAX_TOPK", 5)
    ids, rc = np.arange(100, 120, dtype=np.int64), np.linspace(-2.0, -1.0, 20)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), "c4_", 20, -2.0, ids, rc)
    a, b = _load(tmp_path / "a", "c4_"), _load(tmp_path / "b", "c4_")
    pos = np.load(tmp_path / "a" / "c4_topk_pos.npy")
    assert pos.size == 5 and np.all(np.diff(pos) > 0)
    assert np.array_equal(a["topk_id"], ids[pos.astype(np.int64)]) and np.array_equal(a["topk_rc"], rc[pos.astype(np.int64)])
    assert all(a[n].tobytes() == b[n].tobytes() for n in NAMES)
    assert a["n_violating"][0] == 20 and a["min_rc"][0] == -2.0


@pytest.mark.gpu
def test_device_arm_dump_equals_the_oracle(tmp_path):
    """The timed device pass at 1536 x 1536: the dumped result is bit for bit the oracle's answer on the same
    seeded instance, which bench's own generators rebuild here."""
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    S, K, frac = 1536, 64, 1e-3
    line = _run(tmp_path, "--gpus", "1", "--size", str(S), "--topk", str(K), "--violators", str(frac), "--steps", "3",
                "--warmup", "1", "--no-tree", "--no-cpu", "--no-c4", "--no-manager", "--dump-outputs", str(tmp_path / "d"))
    assert line["config"]["fused"] and line["gpu_launches"] == 3      # one fused launch per timed step, counted
    got = _load(tmp_path / "d")
    import bench
    from oracle import network_oracle as orc
    device = torch.device("cuda", 0)
    P, Q, a = bench.make_points(S, S, device)
    M = bench.make_slab(P, Q, 0, S)
    y = bench.planted_duals(P, Q, a, M, 0, frac, 1)
    cnt, mn, ids, vals = orc.price_summary(orc.reduced_costs_ot(M.cpu().numpy(), y.cpu().numpy()), K)
    assert cnt > K and line["config"]["violating_arcs"] == cnt
    assert got["n_violating"][0] == cnt and got["min_rc"][0] == mn
    assert np.array_equal(got["topk_id"], ids.astype(np.float64)) and got["topk_rc"].tobytes() == vals.tobytes()

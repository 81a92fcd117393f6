"""Row-sharded pricing on REAL ranks: one process per GPU (NCCL), the package's own
`ShardedDensePricer` with every exchange mode, compared with the CPU oracle on the whole matrix.

SURVEY.md section 8(e): the merged top-K is identical for every G because (rc, id) is a strict total
order.  `tests/test_sharded_gloo.py` only covers the host-side partition / block layout (its workers
price with the oracle); this file runs the device kernels, the NVLink peer exchange and the merge.
Needs >= 2 GPUs (`gpurun --gpus 2 -- python -m pytest tests/test_gpu_multirank.py -m gpu`); skipped
on a single-GPU box.
"""
import os
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count() if torch.cuda.is_available() else 0
    except Exception:
        return 0


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _passes(S, D):
    """(name, y) of the passes every rank prices, in order: the double-buffered exchange sees odd and even
    epochs, a converged pass (no violator), massive ties and a pass where most arcs violate."""
    import cases
    s, d, M = cases.ot_points(S, D, 4242)
    ys = [("noise 0.05", cases.planted_duals(M, 11, 0.05)),
          ("converged", cases.planted_duals(M, 11, 0.0) - np.concatenate([np.zeros(S), np.full(D, 1e-3)])),
          ("noise 0.3", cases.planted_duals(M, 12, 0.3)),
          ("noise 0.01", cases.planted_duals(M, 13, 0.01)),
          ("all violate", np.concatenate([np.zeros(S), np.full(D, 5.0)]))]
    return M, ys


def _worker(rank, world, port, exchange, S, D, K, kw):
    import torch
    import torch.distributed as dist
    from oracle import network_oracle as orc
    from smart_crossover.network_methods.sharded import ShardedDensePricer, row_partition
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    device = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=device)
    try:
        M, ys = _passes(S, D)
        row0, S_loc = row_partition(S, world, rank)
        M_loc = torch.from_numpy(np.ascontiguousarray(M[row0:row0 + S_loc])).to(device)
        sp = ShardedDensePricer(M_loc, S, row0, K, exchange=exchange, **kw)
        assert sp.exchange == exchange, f"exchange fell back to {sp.exchange}"
        assert sp.fused == (kw.get("fused") is not False and D % 2 == 0), "fused pass not in the expected state"
        assert sp.fused_merge == (sp.fused and exchange == "ll" and kw.get("fused_merge", True)), "in-kernel merge?"
        for rep in range(2):                       # second sweep replays the captured CUDA graph
            for name, y in ys:
                res = sp.price(y)
                rc = orc.reduced_costs_ot(M, y)
                cnt, mn, ids, vals = orc.price_summary(rc, K)
                tag = f"[{exchange} G={world} K={K} rank={rank} pass '{name}' sweep {rep}]"
                assert res.n_violating == cnt, f"{tag} count {res.n_violating} != {cnt}"
                assert res.min_rc == mn, f"{tag} min {res.min_rc} != {mn}"
                assert np.array_equal(res.topk_id, ids), f"{tag} top-k ids differ"
                assert res.topk_rc.tobytes() == vals.tobytes(), f"{tag} top-k reduced costs differ"
        # the device-resident entry (bench.py's timed arm) returns the same thing
        y = ys[0][1]
        out = sp.enqueue(torch.from_numpy(y).to(device))
        torch.cuda.synchronize()
        cnt, mn, ids, vals = orc.price_summary(orc.reduced_costs_ot(M, y), K)
        n_out = int(out[2].item())
        assert n_out == ids.size and int(out[3].item()) == cnt and int(out[6].item()) == 0
        assert np.array_equal(out[1][:n_out].cpu().numpy(), ids)
        assert out[0][:n_out].cpu().numpy().tobytes() == vals.tobytes()
        dist.barrier()
    finally:
        dist.destroy_process_group()


def _spawn(world, exchange, S, D, K, **kw):
    import torch.multiprocessing as mp
    mp.spawn(_worker, args=(world, _free_port(), exchange, S, D, K, kw), nprocs=world, join=True)


@pytest.mark.skipif(_n_gpus() < 2, reason="needs at least 2 GPUs")
@pytest.mark.parametrize("exchange", ["ll", "p2p", "nccl"])
@pytest.mark.parametrize("K", [64, 1024])
def test_sharded_pricer_on_real_ranks_matches_oracle(exchange, K):
    _spawn(2, exchange, 301, 518, K)


@pytest.mark.skipif(_n_gpus() < 2, reason="needs at least 2 GPUs")
@pytest.mark.parametrize("exchange", ["ll", "nccl"])
def test_sharded_pricer_separate_kernels_on_real_ranks(exchange):
    """The round-1 path (pass begin, pricing, selection, push and merge as separate launches), which prices
    slabs the fused pass cannot take (odd leading dimension, unaligned base), on real ranks."""
    _spawn(2, exchange, 301, 517, 256, fused=False)


@pytest.mark.skipif(_n_gpus() < 2, reason="needs at least 2 GPUs")
@pytest.mark.parametrize("K", [64, 1024])
def test_sharded_pricer_fused_push_with_separate_merge_kernel(K):
    """Fused price + select + push, merge as a kernel of its own (programmatic stream serialisation):
    the path taken when G blocks of K do not fit the in-kernel merge."""
    _spawn(2, "ll", 301, 518, K, fused_merge=False)


@pytest.mark.skipif(_n_gpus() < 2, reason="needs at least 2 GPUs")
def test_sharded_pricer_uneven_rows_and_more_ranks_than_rows_allow():
    """S not divisible by G, and (with every GPU of the box) slabs of a handful of rows."""
    G = min(_n_gpus(), 8)
    _spawn(G, "ll", 8 * G + 3, 700, 256)
    _spawn(2, "ll", 301, 517, 64)                  # odd D: no TMA path, so no fused pass either


@pytest.mark.skipif(_n_gpus() < 4, reason="needs at least 4 GPUs")
@pytest.mark.parametrize("exchange", ["ll", "nccl"])
def test_sharded_pricer_all_gpus(exchange):
    _spawn(min(_n_gpus(), 8), exchange, 1000, 1536, 1024)

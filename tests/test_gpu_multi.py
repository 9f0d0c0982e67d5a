"""N > 1 on real GPUs (needs >= 2 devices; skipped on a 1-GPU box): the peer-store exchange of the C-ABI
(tlc_table_create / tlc_table_attach / tlc_vicinity_pi_exchange, driven by tlc_b200.multi.PeerShardedVicinity) and
the NCCL all-gather path must both leave, on every rank, the table a single-process run produces -- in the caller's
target order, for ragged shards, over several steps (the two halves of the exchange table alternate)."""
import os
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import oracle as orc
from tlc_b200 import _lib as L
from tlc_b200 import api, graphgen as gg, multi


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _problem(step):
    c = gg.make_config("pubmed", scale=0.3, continuous=True)
    labels, ne = gg.relabel_first_appearance(c["edges"])
    csr = gg.build_csr(len(labels), ne, c["kappa"])
    rng = np.random.default_rng(10 + step)
    tg = ne[rng.choice(len(ne), 301 + 7 * step, replace=False)].astype(np.int32)   # odd counts: ragged shards
    tg = np.concatenate([tg, np.array([[-1, 2], [5, 5]], np.int32)])
    return csr, tg


def _worker(rank, world, port, out_path, exchange):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    csr, _ = _problem(0)
    g = api.VicinityGraph(*csr, device=rank)
    flags = L.F_NORM | L.F_EXTENDED
    if exchange == "peer":
        sv = multi.PeerShardedVicinity(g, csr[0], dev, max_rows=1024, hop=2, flags=flags)
    else:
        sv = multi.ShardedVicinity(csr[0], multi.cuda_local_fn(g, dev, hop=2, flags=flags), dev)
    for step in range(3):
        _, tg = _problem(step)
        pi, st = sv.compute(tg)
        torch.cuda.synchronize()
        np.save(out_path % (rank, step), np.concatenate([pi.float().cpu().numpy(), st.float().cpu().numpy()[:, None]], 1))
        dist.barrier()
    g.close()
    dist.destroy_process_group()


@pytest.mark.timeout(900)
@pytest.mark.parametrize("exchange", ["peer", "nccl"])
def test_two_gpu_bench_dumps_the_last_timed_step(tmp_path, exchange):
    """bench.py --dump-outputs on two ranks: rank 0 writes the whole table of the last timed step (both ranks' rows,
    in the step's target order) and it equals the oracle's rows"""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import subprocess
    import sys
    import bench
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    steps, warmup, batch, world = 3, 1, 256, 2
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc_per_node", str(world),
                          os.path.join(root, "bench.py"), "--workload", "cora", "--batch", str(batch), "--steps", str(steps),
                          "--warmup", str(warmup), "--secondary", "0", "--no-cpu-baseline", "--exchange", exchange,
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=800)
    assert out.returncode == 0, out.stderr[-2000:]
    assert sorted(os.listdir(tmp_path)) == ["pi_f32.npy", "status.npy"]
    _, _, ne, csr, perm = bench.make_workload("cora")
    s = warmup + steps - 1
    tg = np.concatenate([bench.batch_targets(ne, perm, s, r, world, batch) for r in range(world)])
    ref = orc.OracleGraph(*csr).run_batch(tg, hop=2, flags=orc.F_NORM)
    assert np.array_equal(np.load(tmp_path / "status.npy"), ref["status"].astype(np.float32))
    den = np.where(ref["pi"] != 0, np.abs(ref["pi"]), 1.0)
    assert float(np.max(np.abs(np.load(tmp_path / "pi_f32.npy") - ref["pi"]) / den)) < 1e-5


@pytest.mark.timeout(600)
@pytest.mark.parametrize("exchange", ["peer", "nccl"])
def test_two_gpu_exchange_matches_oracle(tmp_path, exchange):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    out = str(tmp_path / "rank%d_step%d.npy")
    mp.spawn(_worker, args=(2, _free_port(), out, exchange), nprocs=2, join=True)
    for step in range(3):
        csr, tg = _problem(step)
        ref = orc.OracleGraph(*csr).run_batch(tg, hop=2, flags=orc.F_NORM | orc.F_EXTENDED)
        for r in range(2):
            a = np.load(out % (r, step))
            assert a.shape == (len(tg), 26)
            assert np.array_equal(a[:, 25].astype(np.uint8), ref["status"])
            den = np.where(ref["pi"] != 0, np.abs(ref["pi"]), 1.0)
            assert float(np.max(np.abs(a[:, :25] - ref["pi"]) / den)) < 1e-5

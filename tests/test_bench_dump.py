"""bench.py --dump-outputs: the outputs of the last timed step as <name>.npy files (float32 / float64, at most 64 MB in
all; a larger output is reduced to one seeded sample of rows, the same rows in every file)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _sizes(d):
    return {f: os.path.getsize(os.path.join(d, f)) for f in os.listdir(d)}


def test_dump_small_output_is_written_whole(tmp_path):
    rng = np.random.default_rng(1)
    pi = rng.random((100, 25))
    st = rng.integers(0, 8, 100).astype(np.uint8)
    bench.dump_outputs(str(tmp_path), {"pi": pi, "pi_f32": pi.astype(np.float32), "status": st})
    assert sorted(_sizes(str(tmp_path))) == ["pi.npy", "pi_f32.npy", "status.npy"]
    a = np.load(tmp_path / "pi.npy")
    assert a.dtype == np.float64 and np.array_equal(a, pi)
    s = np.load(tmp_path / "status.npy")
    assert s.dtype == np.float32 and np.array_equal(s, st.astype(np.float32))
    assert np.load(tmp_path / "pi_f32.npy").dtype == np.float32


def test_dump_large_output_is_a_seeded_sample_under_the_limit(tmp_path):
    rows = 300000   # 25 float64 + 25 float32 + 1 status per row: 91 MB before sampling
    pi = np.random.default_rng(2).random((rows, 25))
    arrays = {"pi": pi, "pi_f32": pi.astype(np.float32), "status": (np.arange(rows) % 7).astype(np.uint8)}
    d1, d2 = str(tmp_path / "a"), str(tmp_path / "b")
    bench.dump_outputs(d1, arrays)
    bench.dump_outputs(d2, arrays)
    assert sum(_sizes(d1).values()) <= bench.DUMP_LIMIT
    keep = np.load(os.path.join(d1, "rows.npy"))
    assert keep.dtype == np.float64 and np.all(np.diff(keep) > 0) and 0 < len(keep) < rows
    keep = keep.astype(np.int64)
    assert np.array_equal(np.load(os.path.join(d1, "pi.npy")), pi[keep])
    assert np.array_equal(np.load(os.path.join(d1, "status.npy")), (keep % 7).astype(np.float32))
    for f in _sizes(d1):   # the same sample every time
        assert np.array_equal(np.load(os.path.join(d1, f)), np.load(os.path.join(d2, f)))


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(tmp_path):
    """the dumped rows are the oracle's rows of the LAST timed step's targets (warmup + steps - 1)"""
    import oracle as orc
    steps, warmup, batch = 3, 1, 256
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cora", "--batch", str(batch),
                          "--steps", str(steps), "--warmup", str(warmup), "--secondary", "0", "--no-cpu-baseline",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == steps
    assert sorted(_sizes(str(tmp_path))) == ["pi.npy", "pi_f32.npy", "status.npy"]
    _, _, ne, csr, perm = bench.make_workload("cora")
    tg = bench.batch_targets(ne, perm, warmup + steps - 1, 0, 1, batch)
    ref = orc.OracleGraph(*csr).run_batch(tg, hop=2, flags=orc.F_NORM)
    assert np.array_equal(np.load(tmp_path / "status.npy"), ref["status"].astype(np.float32))
    den = np.where(ref["pi"] != 0, np.abs(ref["pi"]), 1.0)
    assert float(np.max(np.abs(np.load(tmp_path / "pi.npy") - ref["pi"]) / den)) < 1e-5
    assert float(np.max(np.abs(np.load(tmp_path / "pi_f32.npy") - ref["pi"]) / den)) < 1e-5

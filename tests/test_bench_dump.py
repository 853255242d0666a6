"""bench.py --dump-outputs: what the last timed step received, written as .npy so that two builds can be compared
output for output."""
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_small_window_is_whole(tmp_path):
    import torch

    dsts = [torch.randint(0, 256, (100,), dtype=torch.uint8, generator=torch.Generator().manual_seed(j)) for j in range(3)]
    bench.dump_outputs(str(tmp_path / "out"), torch, dsts, [(1, 100)] * 3)
    res = np.load(tmp_path / "out" / "recv_results.npy")
    got = np.load(tmp_path / "out" / "recv_bytes.npy")
    assert res.dtype == np.float64 and res.tolist() == [[1.0, 100.0]] * 3
    assert got.dtype == np.float32 and np.array_equal(got, torch.cat(dsts).numpy())


def test_dump_large_window_is_a_fixed_sample(tmp_path, monkeypatch):
    import torch

    monkeypatch.setattr(bench, "DUMP_SAMPLE", 5000)
    dsts = [torch.randint(0, 256, (1 << 14,), dtype=torch.uint8, generator=torch.Generator().manual_seed(j)) for j in range(4)]
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), torch, dsts, [(1, 1 << 14)] * 4)
    a, b = np.load(tmp_path / "a" / "recv_bytes.npy"), np.load(tmp_path / "b" / "recv_bytes.npy")
    pos = np.sort(np.random.default_rng(0).integers(0, 4 << 14, 5000))
    assert a.dtype == np.float32 and a.shape == (5000,) and np.array_equal(a, b)
    assert np.array_equal(a, torch.cat(dsts).numpy()[pos])


def test_dump_fits_the_output_budget():
    # the default workload (64 x 1 MiB per step) is sampled; the sample and the results stay under 64 MB
    assert bench.WINDOW * bench.MSG_BYTES > bench.DUMP_SAMPLE
    assert bench.DUMP_SAMPLE * 4 + bench.WINDOW * 2 * 8 <= 64 << 20


@pytest.mark.gpu
def test_bench_dump_is_the_last_window_sent(tmp_path):
    """At N == 1 the last timed step receives its own sources: the seeded set (steps - 1) % POOL_SETS.  With 3 warm-up
    and 4 timed steps that is set 3, which only the timed steps fill."""
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    steps, window, msg = 4, 8, 4096
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "3", "--msg-bytes", str(msg),
           "--window", str(window), "--no-sweep", "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=280, env=dict(os.environ, STARWAY_QUIET="1"))
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    assert np.load(tmp_path / "recv_results.npy").tolist() == [[bench.TAG, msg]] * window
    g = torch.Generator(device="cuda").manual_seed(0xB200)
    sets = [torch.cat([torch.randint(0, 256, (msg,), dtype=torch.uint8, device="cuda", generator=g) for _ in range(window)])
            for _ in range(bench.POOL_SETS)]
    got = np.load(tmp_path / "recv_bytes.npy")
    assert got.dtype == np.float32 and np.array_equal(got, sets[(steps - 1) % bench.POOL_SETS].cpu().numpy())

"""bench.py --dump-outputs: the files are bounded, reproducible and sampled in logical order (CPU), and on the GPU they
hold what the timed step computed -- checked against the oracle on the same seeded inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
from conftest import assert_grad_parity, assert_terms_parity
from oracle import torch_oracle as TO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TERMS = ["l1", "gd", "ssim", "ce", "tv"]


def test_dump_outputs_is_bounded_reproducible_and_in_logical_order(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 8000)
    shape = (2, 20, 30, 40)
    big = torch.arange(np.prod(shape), dtype=torch.float32).reshape(shape).contiguous(memory_format=torch.channels_last)
    small = torch.arange(8, dtype=torch.float32)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"loss": small, "d_src_layout": big})
    total = sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a"))
    assert sorted(os.listdir(tmp_path / "a")) == ["d_src_layout.npy", "loss.npy"] and total <= 8000
    for name in ("loss", "d_src_layout"):
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, b)
    assert np.array_equal(np.load(tmp_path / "a" / "loss.npy"), small.numpy())
    sample = np.load(tmp_path / "a" / "d_src_layout.npy")
    # every element holds its own logical (NCHW) flat index: a sample in logical order is sorted, one in memory order not
    assert sample.ndim == 1 and sample.size > 100 and np.all(np.diff(sample) >= 0) and sample[-1] < big.numel()


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(tmp_path):
    """c1 with --steps 3: exactly three timed steps, and the last one ran on the first of the two alternating input sets
    (seed 1024); its loss vector and gradients are written whole and agree with the oracle at the parity bar."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c1", "--steps", "3", "--warmup", "1",
                          "--no-sweep", "--no-train", "--no-aux", "--no-eager", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 3 and line["config"]["replays_per_step"] == 1
    N, H, W, K, sigma, far, _ = bench.WORKLOADS["c1"]
    d = bench.make_inputs(N, H, W, K, sigma, far, "f32", None, seed=1024)
    args = (d["src_rgb"], d["src_layout"], d["flow"], d["tgt_rgb"], d["tgt_label"])
    ref32 = TO.warp_loss_fwd_bwd(*args, w_tv=0.5)
    ref64 = TO.warp_loss_fwd_bwd(*args, w_tv=0.5, dtype=torch.float64)
    loss = np.load(tmp_path / "loss.npy")
    assert_terms_parity(loss[:5], [ref32["terms"][k].item() for k in TERMS], [ref64["terms"][k].item() for k in TERMS], 1e-5)
    for k in ("d_flow", "d_src_rgb", "d_src_layout"):
        got = np.load(tmp_path / f"{k}.npy")
        assert got.shape == tuple(ref32[k].shape), k
        assert_grad_parity(got, ref32[k], ref64[k], 1e-5, k)

"""bench.py as a user runs it: argument checks (CPU tier) and, on the GPU, --dump-outputs -- the headline layer's
output of the last timed step, written as float32 .npy, is the GCN layer of the seeded inputs (fp64 oracle)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import rel_gate
from gnnagg import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")


def test_bench_rejects_zero_steps(tmp_path):
    p = subprocess.run([sys.executable, BENCH, "--steps", "0"], cwd=tmp_path, capture_output=True, text=True, timeout=120)
    assert p.returncode == 2 and "--steps" in p.stderr


def test_output_sample_is_fixed_and_within_budget():
    import torch

    import bench

    Y = torch.arange(1000 * 8, dtype=torch.float32).reshape(1000, 8)
    whole, how = bench.output_sample(Y, 1000 * 8 * 4)
    assert np.array_equal(whole, Y.numpy()) and how == "all 1000 rows"
    a, _ = bench.output_sample(Y, 100 * 8 * 4 + 31)
    b, _ = bench.output_sample(Y.clone(), 100 * 8 * 4 + 31)
    assert a.shape == (100, 8) and a.dtype == np.float32 and np.array_equal(a, b)
    rows = a[:, 0].astype(np.int64) // 8
    assert np.all(np.diff(rows) > 0) and np.array_equal(a, Y.numpy()[rows])


@pytest.mark.gpu
def test_bench_dump_outputs_is_the_layer_output(orc, cuda, tmp_path):
    import torch

    out_dir = tmp_path / "out"
    cmd = [sys.executable, BENCH, "--gpus", "1", "--steps", "4", "--warmup", "3", "--workload", "arxiv_gcn_layer_32",
           "--c5", "0", "--ref-kernels", "0", "--cpu-seconds", "0.2", "--dump-outputs", str(out_dir)]
    p = subprocess.run(cmd, cwd=tmp_path, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-3000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["steps"] == 4
    n, m = synth.shape_of("arxiv")
    assert sorted(os.listdir(out_dir)) == ["H.npy"]
    H = np.load(out_dir / "H.npy")
    assert H.dtype == np.float32 and H.shape == (n, 32)  # 21.7 MB: the whole output, no sampling
    assert line["outputs_dumped"]["files"] == ["H.npy"] and line["outputs_dumped"]["H"]["shape"] == [n, 32]
    # the inputs bench.py builds for this workload at N = 1, restated here so that the fp64 check does not run through
    # the code under test: Workload.__init__ in bench.py is the source of truth (graph seed 123, X seed 123 + rank,
    # W seed 7 scaled by 1/sqrt(F)); if its seeding changes, change it here too or this parity check fails
    ptr, idx = synth.rmat_csr(n, m, seed=123, device=cuda)
    val = synth.gcn_norm_val(ptr, idx)
    X = torch.randn((n, 32), device=cuda, generator=torch.Generator(device=cuda).manual_seed(123))
    W = torch.randn((32, 32), device=cuda, generator=torch.Generator(device=cuda).manual_seed(7)) / 32 ** 0.5
    _, h64, scale = orc.gcn_layer_f64(ptr.cpu().numpy(), idx.cpu().numpy(), val.cpu().numpy(), X.cpu().numpy(),
                                      W.cpu().numpy())
    assert rel_gate(H, h64, scale, 1e-5)[0] == 0

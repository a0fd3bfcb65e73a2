"""bench.py --dump-outputs: the outputs of the last timed step are written as .npy files, equal from run to run (seeded
inputs, whatever --steps is) and equal to the oracle on the same inputs.  D is above bench.DUMP_COLUMNS, so `out` is
the seeded column sample."""
from __future__ import annotations

import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

import bench
from conftest import ATOL, RTOL
from oracle import bde_oracle as O

ROOT = Path(__file__).resolve().parent.parent
D = 1_200_000


def run_bench(steps, dump):
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
                          "--skip-extras", "--d-per-gpu", str(D), "--dump-outputs", str(dump)],
                         capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-4000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["gpu_launches"] == 2 * steps   # K1 (+K1b) and K2 per timed step
    files = sorted(p.name for p in dump.iterdir())
    assert files == ["bandwidth_info.npy", "kernel_A.npy", "kernel_K.npy", "median_sel.npy", "out.npy", "pair_dist.npy"]
    assert sum(p.stat().st_size for p in dump.iterdir()) <= 64 << 20
    return {f[:-4]: np.load(dump / f) for f in files}


@pytest.mark.gpu
def test_dump_outputs_are_reproducible_and_match_the_oracle(tmp_path):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    a = run_bench(3, tmp_path / "a")
    b = run_bench(1, tmp_path / "b")
    for name, arr in a.items():
        assert arr.dtype in (np.float32, np.float64), name
        np.testing.assert_array_equal(arr, b[name], err_msg=name)
    n = bench.N_PARTICLES
    X, G = (t.cpu() for t in bench.make_inputs(n, D, 0, torch.device("cuda")))
    d = O.svgd_pairdist(X, chunk=1 << 16)
    bw = O.svgd_bandwidth(d, bench.L2_REG, bench.KERNEL_GRAD_SCALE, bench.DATASET_SIZE)
    np.testing.assert_allclose(a["pair_dist"], d.numpy(), rtol=2e-6, atol=1e-12)
    assert tuple(a["median_sel"].astype(int)) == bw["sel"]
    np.testing.assert_allclose(a["bandwidth_info"], [bw["h"], bw["median"], bw["d_lo"], bw["d_hi"]], rtol=2e-6)
    np.testing.assert_allclose(a["kernel_K"], bw["K"].numpy(), rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(a["kernel_A"], bw["A"].numpy(), rtol=RTOL, atol=ATOL)
    idx = torch.from_numpy(np.sort(np.random.default_rng(0).choice(D, bench.DUMP_COLUMNS, replace=False)))
    assert a["out"].shape == (n, bench.DUMP_COLUMNS)
    np.testing.assert_allclose(a["out"], O.svgd_apply(X[:, idx], G[:, idx], bw["K"], bw["A"]).numpy(), rtol=RTOL, atol=ATOL)

"""SVGD with 33 to 64 particles on the GPU: K1 (+K1b), K2 and the whole step at n in {24, 33, 48, 64} x D = 2e7.

n = 24 runs the generic runtime-n kernels (context); 33..64 the particle-tiled kernels of csrc/svgd_many.cu.  The
working set (X, G, out: 12 n D bytes, >= 5.8 GB) is far above the 126 MB L2, so every timed pass streams from HBM.
CUDA events around `--reps` launches after `--warmup` launches of every shape.  Rates are algorithmic: K1 reads
4 n D bytes, K2 reads 8 n D and writes 4 n D, the step moves 16 n D; the copy rate is a device-to-device copy of
an [n, D] fp32 matrix (8 n D bytes moved) timed the same way, in the same run.  The eager reference-order step
(oracle.svgd_step_reference_order in fp32, the reference's own ATen ops) runs on the same GPU at the same shapes,
with the same warm-up and repetition counts.

    python tools/exp_many_particles.py --out profiles/r03_many_particles.jsonl
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from beyond_deep_ensembles_b200 import ops  # noqa: E402
from oracle import bde_oracle as O  # noqa: E402

BW = (0.01, 1.0, 768.0)


def time_ms(fn, warmup: int, reps: int) -> float:
    for _ in range(warmup):
        fn()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0.record()
    for _ in range(reps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / reps


def gpu_identity() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--ns", default="24,33,48,64")
    ap.add_argument("--D", type=int, default=20_000_000)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    D = a.D
    rows = [dict(kind="identity", **gpu_identity())]
    print(json.dumps(rows[0]), flush=True)
    for n in map(int, a.ns.split(",")):
        g = torch.Generator(device="cuda").manual_seed(n)
        scale = 0.05 * (1 + 0.1 * torch.arange(n, dtype=torch.float32, device="cuda")).unsqueeze(1)
        X = scale * torch.randn(n, D, generator=g, device="cuda")
        G = 1e-3 * torch.randn(n, D, generator=g, device="cuda")
        out = torch.empty_like(X)
        sc = ops.SvgdScratch.allocate(n, "cuda")
        copy_ms = time_ms(lambda: out.copy_(X), a.warmup, a.reps)
        copy_gbs = 8 * n * D / copy_ms / 1e6
        k1_ms = time_ms(lambda: ops.svgd_pairdist_bandwidth(X, sc, *BW), a.warmup, a.reps)
        k2_ms = time_ms(lambda: ops.svgd_apply(X, G, out, sc), a.warmup, a.reps)
        step_ms = time_ms(lambda: ops.svgd_step(X, G, out, sc, *BW), a.warmup, a.reps)
        eager_ms = time_ms(lambda: O.svgd_step_reference_order(X, G, *BW, dtype=torch.float32), a.warmup, a.reps)
        row = dict(kind="svgd", n=n, D=D, copy_ms=copy_ms, copy_GBs=copy_gbs,
                   k1_ms=k1_ms, k1_GBs=4 * n * D / k1_ms / 1e6,
                   k2_ms=k2_ms, k2_GBs=12 * n * D / k2_ms / 1e6,
                   step_ms=step_ms, step_GBs=16 * n * D / step_ms / 1e6,
                   eager_reference_ms=eager_ms, speedup_vs_eager=eager_ms / step_ms,
                   warmup=a.warmup, reps=a.reps)
        for k in ("k1", "k2", "step"):
            row[f"{k}_frac_of_copy"] = row[f"{k}_GBs"] / copy_gbs
        rows.append(row)
        print(json.dumps(row), flush=True)
        del X, G, out
        torch.cuda.empty_cache()
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text("".join(json.dumps(r) + "\n" for r in rows))


if __name__ == "__main__":
    main()

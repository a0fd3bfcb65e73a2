#!/usr/bin/env python
"""bench.py — optimizer-step time and HBM GB/s of the posterior-update hot path.

Headline workload (BASELINE.json configs[4], the sweep the north-star target is quoted on):
one SVGD posterior update over n=10 particles x D=100 M parameters PER GPU (weak scaling:
every rank holds a [10, D] column slice of X / G / out; only the 10x10 fp64 partial distance
matrix is all-reduced).  A step is K1 (+K1b) -> K2 over data resident in HBM.

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference        # the reference's CPU path (oracle port) on host cores
    python bench.py --gpus 1 --steps 20 --warmup 3 --dump-outputs DIR   # also write the last step's outputs to DIR

Prints ONE JSON line on rank 0 (everything else goes to stderr).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_PARTICLES = 10
D_PER_GPU = 100_000_000
L2_REG, KERNEL_GRAD_SCALE, DATASET_SIZE = 0.01, 1.0, 50000.0
CPU_SAMPLE_D = 10_000_000
METRIC = "svgd_posterior_update_algorithmic_GBps"
DUMP_COLUMNS = 1 << 20   # columns of `out` --dump-outputs writes: n x 2^20 fp32 = 40 MB at n = 10, inside its 64 MB cap


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# --------------------------------------------------------------------------------------
# clocks (sampled DURING the timed region)
# --------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, index: int):
        self.samples, self.reasons, self.sm_max = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # noqa: BLE001
            log(f"[bench] NVML unavailable: {e}")
            self.nv = None

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                get = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
                mask = get(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.005)

    def __enter__(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thr is not None:
            self._thr.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.sm_max,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# --------------------------------------------------------------------------------------
# CPU baseline / reference arm: the UNMODIFIED reference SVGDOptimizer.step (oracle/_ref, staged by
# oracle/install_ref.py) on the host cores; the oracle's port of its op sequence only if oracle/_ref is missing
# --------------------------------------------------------------------------------------
def synth_host(n, D, seed=0):
    g = torch.Generator().manual_seed(seed)
    X = torch.randn(n, D, generator=g)
    X *= (0.05 * (1 + 0.1 * torch.arange(n, dtype=torch.float32))).unsqueeze(1)
    G = torch.randn(n, D, generator=g) * 1e-3
    return X, G


REF_INCLUDES = ("whole SVGDOptimizer.step of the reference (src/algos/svgd.py:65-105) with free closures: per-particle "
                "_use_particle / grad clone, gather into [n, D] (parameters_to_vector + stack), prior term, rbf (cdist, "
                "quantile, exp, matmul), phi, per-particle scatter (slice + clone) and n plain-SGD base-optimizer steps")


def cpu_reference_run(steps: int, warmup: int, D: int = CPU_SAMPLE_D, threads: int | None = None):
    """Times the posterior-update path of the reference on the host in fp32 with every host thread torch will use
    (or `threads`).  Returns (GB/s, ms/step, threads, kind, D): kind "reference" = the unmodified SVGDOptimizer.step
    from oracle/_ref driven by oracle/ref_driver.py; "port" = oracle.svgd_step_reference_order (same ATen op
    sequence, no gather / scatter / base optimizer) when the staged reference is absent."""
    from oracle import install_ref
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    if install_ref.available():
        from oracle import ref_driver
        X, G = ref_driver.synth(N_PARTICLES, D, "cpu")
        job = ref_driver.ReferenceSvgdJob(X, G, L2_REG, KERNEL_GRAD_SCALE, DATASET_SIZE)
        t0 = time.perf_counter()
        job.step()                                   # first warm-up step, also the size probe
        first = time.perf_counter() - t0
        if first * (steps + warmup) > 240.0 and D > 2_000_000:   # keep the whole run inside a few minutes
            return cpu_reference_run(steps, warmup, D // 5, threads)
        ms = ref_driver.time_reference_steps(job, max(1, steps), max(0, warmup - 1))
        kind = "reference"
    else:
        from oracle import bde_oracle as O
        X, G = synth_host(N_PARTICLES, D)
        for _ in range(max(1, warmup)):
            O.svgd_step_reference_order(X, G, L2_REG, KERNEL_GRAD_SCALE, DATASET_SIZE)
        t0 = time.perf_counter()
        for _ in range(max(1, steps)):
            O.svgd_step_reference_order(X, G, L2_REG, KERNEL_GRAD_SCALE, DATASET_SIZE)
        ms = 1e3 * (time.perf_counter() - t0) / max(1, steps)
        kind = "port"
    gbs = 16.0 * N_PARTICLES * D / (ms * 1e-3) / 1e9
    return gbs, ms, torch.get_num_threads(), kind, D


def cpu_sample_text(kind, D, steps):
    what = ("the unmodified reference SVGDOptimizer.step (oracle/_ref/src/algos/svgd.py driven by oracle/ref_driver.py: "
            + REF_INCLUDES + ")") if kind == "reference" else \
           "oracle.svgd_step_reference_order (port of the reference's ATen op sequence; no gather / scatter / base optimizer)"
    return (f"n={N_PARTICLES} x D={D} fp32 on the host ({D / D_PER_GPU:.0%} of one GPU's columns; the rate is per byte, so "
            f"the sample size does not enter the metric), {steps} timed steps of {what}")


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = args.steps, max(1, args.warmup)   # same steps / warm-up as the GPU arm
    gbs, ms, threads, kind, D = cpu_reference_run(steps, warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": gbs, "unit": "GB/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": gbs, "unit": "GB/s", "cores": threads, "kind": kind, "sample": cpu_sample_text(kind, D, steps)},
        "e2e": {"value": gbs, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def workload_config(n_gpus):
    return {
        "workload": "MultiX-SVGD optimizer-step sweep point: n=10 particles x D=100M params per GPU, D-sharded",
        "particles": N_PARTICLES, "D_per_gpu": D_PER_GPU, "D_total": D_PER_GPU * n_gpus,
        "l2_reg": L2_REG, "dataset_size": DATASET_SIZE, "kernel_grad_scale": KERNEL_GRAD_SCALE,
        "algorithmic_bytes_per_step_per_gpu": 16 * N_PARTICLES * D_PER_GPU,
        "l2_flush": "inputs (12 GB per GPU) are larger than the 126 MB L2",
        "parallelism": f"D-shard x{n_gpus}; only the 10x10 fp64 partial distances cross NVLink (summed inside K1's tail "
                       "over peer memory, or by one NCCL all-reduce)",
    }


def eager_cuda_reference(dev, D=None, steps=3):
    """The kernel-for-kernel competitor of SURVEY.md §8(d): the same unmodified reference class, eager PyTorch on THIS
    GPU (device-resident inputs, wall clock bracketed by synchronize).  None if oracle/_ref is not staged."""
    from oracle import install_ref
    if not install_ref.available():
        return None
    from oracle import ref_driver
    D = D or D_PER_GPU
    try:
        torch.cuda.reset_peak_memory_stats(dev)
        X, G = ref_driver.synth(N_PARTICLES, D, dev)
        job = ref_driver.ReferenceSvgdJob(X, G, L2_REG, KERNEL_GRAD_SCALE, DATASET_SIZE)
        del X
        ms = ref_driver.time_reference_steps(job, steps, 1, sync=torch.cuda.synchronize)
        peak_gb = torch.cuda.max_memory_allocated(dev) / 1e9
        res = {"ms_per_step": ms, "GBps": 16.0 * N_PARTICLES * D / (ms * 1e-3) / 1e9, "steps": steps, "kind": "reference",
               "what": f"oracle/_ref SVGDOptimizer.step, eager PyTorch on the same GPU, n={N_PARTICLES} x D={D}: " + REF_INCLUDES,
               "peak_device_memory_GB": peak_gb}
        log(f"[bench] reference eager on this GPU: {ms:.2f} ms/step")
        del job, G
    except Exception as e:  # noqa: BLE001
        log(f"[bench] eager_cuda reference failed: {e}")
        res = {"error": str(e)}
    torch.cuda.empty_cache()
    return res


# --------------------------------------------------------------------------------------
# GPU helpers
# --------------------------------------------------------------------------------------
def time_kernel(fn, iters, warmup, flush=None):
    """Mean device ms of fn() (CUDA events on the current stream).

    Working set larger than L2 (flush=None): `iters` back-to-back launches between one event pair,
    as inside a real optimizer step.  Working set smaller than L2: every launch is timed on its
    own after overwriting a buffer larger than L2."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if flush is None:
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / iters
    total = 0.0
    for _ in range(iters):
        flush.zero_()
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        total += e0.elapsed_time(e1)
    return total / iters


def other_paths(ops, peak_gbs, dev):
    """The other kernels of the path at their named configs (SURVEY.md §8d), device-resident,
    L2 flushed between iterations when the working set is smaller than L2."""
    res = {}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    copy_cache = {}

    def same_size_copy(nbytes):
        """GB/s of a plain device copy that moves the SAME number of bytes (half read, half written): a 0.1 ms kernel
        cannot reach the rate MEASURED_PEAKS.json quotes for a 4 GB copy (launch ramp and tail are ~8 % of it)."""
        key = int(nbytes) >> 20
        if key not in copy_cache:
            a = torch.empty(max(int(nbytes) // 8, 1), dtype=torch.float32, device=dev)
            b = torch.empty_like(a)
            ms = time_kernel(lambda: b.copy_(a), 20, 3, flush if nbytes < (200 << 20) else None)
            copy_cache[key] = 8.0 * a.numel() / (ms * 1e-3) / 1e9
            del a, b
        return copy_cache[key]

    def rec(name, ms, nbytes, cfg, size_ref=False):
        gbs = nbytes / (ms * 1e-3) / 1e9
        res[name] = {"ms": ms, "GBps": gbs, "frac_of_measured_peak": gbs / peak_gbs, "algorithmic_bytes": nbytes,
                     "config": cfg}
        extra = ""
        if size_ref:
            ref = same_size_copy(nbytes)
            res[name].update(same_size_copy_GBps=ref, frac_of_same_size_copy=gbs / ref)
            extra = f", {gbs / ref:.2%} of a torch copy of the same {nbytes / 1e6:.0f} MB"
        log(f"[bench] {name}: {ms:.4f} ms  {gbs:.0f} GB/s  ({gbs / peak_gbs:.2%} of measured copy peak{extra})")

    g = torch.Generator(device=dev).manual_seed(1)
    # C3 SWAG, ResNet-50 + fc182, K = 10
    D, K = 23_880_950, 10
    Dp = (D + 63) // 64 * 64
    theta = torch.randn(Dp, device=dev, generator=g) * 0.05
    mean = theta + torch.randn(Dp, device=dev, generator=g) * 0.01
    sq = mean * mean + 1e-4
    ring = torch.randn(K, Dp, device=dev, generator=g) * 0.01
    out = torch.empty(Dp, device=dev)
    u = [0]

    def swag_upd():
        u[0] += 1
        ops.swag_update(theta, mean, sq, ring[(u[0] - 1) % K], u[0])

    rec("swag_update", time_kernel(swag_upd, 20, 3), 24 * Dp, f"ResNet-50 D={D}, K={K}", size_ref=True)
    rec("swag_sample", time_kernel(lambda: ops.swag_sample(mean, sq, ring, 3, out, seed=1, stream_id=2), 20, 3),
        4 * (K + 3) * Dp, f"ResNet-50 D={D}, K={K}, Philox noise", size_ref=True)
    # f3: 16 draws from the same posterior in one pass (DeepEnsemble.predict) vs 16 single launches
    S = 16
    outs = torch.empty(S, Dp, device=dev)
    # (A/B on B200 of the draws per pass, bde_tune("swag_batch"): 16 -> 0.995 ms, 8 -> 1.034 ms, 4 -> 1.234 ms)
    ms_b = time_kernel(lambda: ops.swag_sample_batch(mean, sq, ring, 3, outs, seed=1, stream_id=2), 10, 3)
    rec("swag_sample_batch16", ms_b, 4 * (K + 2 + S) * Dp,
        f"ResNet-50 D={D}, K={K}, {S} draws in one pass (reads the moments once; bound by the {S} x D Philox normals, "
        f"not by HBM); {S} single launches move {4 * (K + 3) * S} x D bytes and take {S * res['swag_sample']['ms']:.3f} ms")
    del theta, mean, sq, ring, out, outs
    # C4b iVON, DistilBERT + head
    D = 66_955_010
    Dp = (D + 63) // 64 * 64
    mean = torch.randn(Dp, device=dev, generator=g) * 0.05
    prec = torch.rand(Dp, device=dev, generator=g) * 1e-4 + 10.0 / 269038   # mid-training state: all non-trivial
    mom = torch.randn(Dp, device=dev, generator=g) * 1e-4
    dsum = torch.randn(Dp, device=dev, generator=g) * 0.3
    acc = torch.randn(Dp, device=dev, generator=g) * 2e-5   # small enough that the precision stays positive over the timed calls
    theta = torch.zeros(Dp, device=dev)
    grad = torch.randn(Dp, device=dev, generator=g) * 1e-3
    kw = dict(n_eff=269038.0)
    rec("ivon_sample", time_kernel(lambda: ops.ivon_sample(mean, prec, dsum, theta, first=False, seed=1, stream_id=3, **kw), 20, 3),
        20 * Dp, f"DistilBERT D={D}, Philox noise", size_ref=True)
    rec("ivon_accumulate", time_kernel(lambda: ops.ivon_accumulate(acc, grad, first=False), 20, 3), 12 * Dp, f"D={D}", size_ref=True)
    # f3: 16 MC draws in one pass (DeepEnsemble.predict on an iVON member): mean / precision read once, delta_sum RMW once
    S = 16
    outs = torch.empty(S, Dp, device=dev)
    ms_b = time_kernel(lambda: ops.ivon_sample_batch(mean, prec, dsum, outs, first=False, seed=1, stream_id=3, **kw), 10, 3)
    rec("ivon_sample_batch16", ms_b, 4 * (4 + S) * Dp,
        f"DistilBERT D={D}, {S} draws in one pass (fast kernel: unrolled independent Philox chains; bound by the {S} x D "
        f"normals, not by HBM); {S} single launches move {20 * S} x D bytes and take {S * res['ivon_sample']['ms']:.3f} ms")
    del outs
    # the two timing loops above accumulated 23 samples / gradients into dsum and acc: put a
    # mid-training state back so that the update runs on realistic magnitudes (finite everywhere)
    dsum.normal_(0.0, 0.3, generator=g)
    acc.normal_(0.0, 2e-5, generator=g)
    step = [0]

    def ivon_upd():
        step[0] += 1
        ops.ivon_update(acc, dsum, mean, mom, prec, mc_samples=2, step=100 + step[0], lr=1e-5, beta1=0.9, beta2=0.999,
                        prior_prec=10.0, n_eff=269038.0, tempering=1.0, damping=1e-3)

    rec("ivon_update", time_kernel(ivon_upd, 20, 3), 32 * Dp, f"DistilBERT D={D}", size_ref=True)
    del mean, prec, mom, dsum, theta, acc, grad
    # C4a BBB last layer: P = 592,130 Gaussian weights; deterministic DistilBERT body 66.36 M
    P = 592_130
    Pp = (P + 63) // 64 * 64
    mu = torch.randn(Pp, device=dev, generator=g) * 0.1
    rho = torch.full((Pp,), -3.0, device=dev)
    w, gmu, grho = (torch.zeros(Pp, device=dev) for _ in range(3))
    val = torch.zeros((), dtype=torch.float64, device=dev)
    ws = ops.value_workspace(dev)
    rec("gauss_sample_fwd", time_kernel(lambda: ops.gauss_sample_fwd(mu, rho, w, seed=1, stream_id=4), 20, 3, flush),
        12 * Pp, f"BBB head P={P} (launch-bound)")
    rec("gauss_sample_bwd", time_kernel(lambda: ops.gauss_sample_bwd(w, rho, grho, seed=1, stream_id=4), 20, 3, flush),
        16 * Pp, f"BBB head P={P} (launch-bound)")
    rec("kl_gauss_value_and_grad",
        time_kernel(lambda: ops.kl_gauss(mu, rho, 0.0, 1.0, value=val, grad_mu=gmu, grad_rho=grho, accumulate=True, ws=ws), 20, 3, flush),
        24 * Pp, f"BBB head P={P} (launch-bound)")
    # f4: BBBLinear local-reparameterisation forward of the Civil head (768 x 768, batch 16) as one tcgen05 kernel, next to
    # the reference layer's eager CUDA branch (bbb_layers.py:66-79: stacks, pow, clamps, softplus, baddbmm, sqrt, noise)
    try:
        from beyond_deep_ensembles_b200 import bbb_layers
        xb = torch.randn(16, 768, device=dev, generator=g)
        wmu = 0.1 * torch.randn(768, 768, device=dev, generator=g)
        wrho = torch.full((768, 768), -3.0, device=dev)
        bmu, brho = torch.zeros(768, device=dev), torch.full((768,), -3.0, device=dev)

        def ref_layer():
            sw, sb = torch.nn.functional.softplus(wrho), torch.nn.functional.softplus(brho)
            bin_ = torch.stack((xb, (xb ** 2).clamp(min=1e-4)))
            bmat = torch.stack((wmu.transpose(0, 1), (sw.transpose(0, 1) ** 2).clamp(min=1e-4)))
            badd = torch.stack((bmu.expand((16, 768)), (sb ** 2).clamp(min=1e-4).expand((16, 768))))
            bo = torch.baddbmm(badd, bin_, bmat)
            return bo[0] + torch.sqrt(bo[1]) * torch.empty_like(bo[0]).normal_(0, 1)

        ms_f = time_kernel(lambda: ops.bbb_linear_fwd(xb, wmu, wrho, bmu, brho, seed=1, stream_id=2, workspace=bbb_layers._workspace), 30, 5, flush)
        ms_r = time_kernel(ref_layer, 30, 5, flush)
        res["bbb_linear_fwd_civil_head"] = {
            "fused_tcgen05_ms": ms_f, "reference_eager_cuda_ms": ms_r, "speedup": ms_r / ms_f,
            "config": "BBBLinear(768, 768), batch 16, fp32: one tcgen05 kernel (exact 3-way tf32 split, TMEM accumulators, "
                      "tensor-map TMA) vs the reference layer's own eager CUDA branch incl. torch.baddbmm; L2 flushed"}
        log(f"[bench] bbb_linear_fwd (Civil head): fused {1e3 * ms_f:.1f} us vs reference eager {1e3 * ms_r:.1f} us ({ms_r / ms_f:.2f}x)")
        # Rank1Linear.forward (rank1.py:50-64) at the same head: both samples + x * s + product + * r + bias in one launch
        smu, srho = torch.ones(768, device=dev), torch.full((768,), -3.0, device=dev)

        def ref_rank1():
            s1 = smu + torch.empty_like(smu).normal_(0, 1) * torch.nn.functional.softplus(srho)
            r1 = smu + torch.empty_like(smu).normal_(0, 1) * torch.nn.functional.softplus(srho)
            o1 = torch.nn.functional.linear(xb * s1, wmu) * r1
            o1 += bmu.unsqueeze(0)
            return o1

        ms_f1 = time_kernel(lambda: ops.rank1_linear_fwd(xb, wmu, smu, srho, smu, srho, bmu, seed=1, stream_id_s=2, stream_id_r=3,
                                                         workspace=bbb_layers._workspace), 30, 5, flush)
        ms_r1 = time_kernel(ref_rank1, 30, 5, flush)
        res["rank1_linear_fwd_civil_head"] = {
            "fused_tcgen05_ms": ms_f1, "reference_eager_cuda_ms": ms_r1, "speedup": ms_r1 / ms_f1,
            "config": "Rank1Linear(768, 768), batch 16, fp32: one tcgen05 kernel vs the reference layer's expression in eager "
                      "PyTorch (2 samples, mul, F.linear, mul, add); L2 flushed"}
        log(f"[bench] rank1_linear_fwd (Civil head): fused {1e3 * ms_f1:.1f} us vs reference eager {1e3 * ms_r1:.1f} us ({ms_r1 / ms_f1:.2f}x)")
        del xb, wmu, wrho
    except Exception as e:  # noqa: BLE001
        res["bbb_linear_fwd_civil_head"] = {"error": str(e)}
    Dd = 66_362_880
    body = torch.randn(Dd, device=dev, generator=g) * 0.02
    gbody = torch.zeros(Dd, device=dev)
    rec("l2_value_and_grad",
        time_kernel(lambda: ops.l2_term(body, 0.01, value=val, grad=gbody, accumulate=True, ws=ws), 20, 3),
        12 * Dd, f"DistilBERT body D={Dd}")
    del body, gbody
    # f1: K2 fused with the base optimizer (shared state, one step per particle), n = 10 x D = 1e8,
    # next to what the reference's structure costs on the same GPU: K2 + n x torch.optim step()
    nf, Df = N_PARTICLES, D_PER_GPU
    Xf = torch.randn(nf, Df, device=dev, generator=g)
    Xf *= (0.05 * (1 + 0.1 * torch.arange(nf, device=dev, dtype=torch.float32))).unsqueeze(1)
    Gf = torch.randn(nf, Df, device=dev, generator=g) * 1e-3
    scf = ops.SvgdScratch.allocate(nf, dev)
    ops.svgd_pairdist_bandwidth(Xf, scf, L2_REG, KERNEL_GRAD_SCALE, DATASET_SIZE)
    buf, buf2, olast = (torch.zeros(Df, device=dev) for _ in range(3))
    sgd_kw = dict(lr=1e-4, momentum=0.9, nesterov=True, weight_decay=3e-4)
    rec("svgd_apply_fused_sgd",
        time_kernel(lambda: ops.svgd_apply_sgd(Xf, Gf, scf, buf, buf_initialized=True, out_last=olast, **sgd_kw), 10, 3),
        (12 * nf + 12) * Df, f"n={nf} x D={Df}: K2 + {nf} SGD(momentum, nesterov, wd) steps in one pass, X in place")
    st0 = [0]

    def fused_adam():
        ops.svgd_apply_adam(Xf, Gf, scf, buf, buf2, step0=st0[0], lr=1e-5, out_last=olast)
        st0[0] += nf

    rec("svgd_apply_fused_adam", time_kernel(fused_adam, 10, 3), (12 * nf + 20) * Df,
        f"n={nf} x D={Df}: K2 + {nf} Adam steps in one pass, X in place")
    # training-step form: the same pass also yields the NEXT step's pair distances + K1b, so a steady-state
    # SVGD training step (posterior update + n base-optimizer steps) is this ONE launch
    nk = ops.NextKernel(True, L2_REG, KERNEL_GRAD_SCALE, DATASET_SIZE)
    rec("svgd_train_step_fused_sgd",
        time_kernel(lambda: ops.svgd_apply_sgd(Xf, Gf, scf, buf, buf_initialized=True, out_last=olast, next_kernel=nk, **sgd_kw), 10, 3),
        (12 * nf + 12) * Df, f"n={nf} x D={Df}: K2 + {nf} SGD steps + next step's K1/K1b in one pass "
        f"(bytes moved; the reference structure needs {16 * nf + 12 * nf} x D bytes for the same work)")

    def train_adam():
        ops.svgd_apply_adam(Xf, Gf, scf, buf, buf2, step0=st0[0], lr=1e-5, out_last=olast, next_kernel=nk)
        st0[0] += nf

    rec("svgd_train_step_fused_adam", time_kernel(train_adam, 10, 3), (12 * nf + 20) * Df,
        f"n={nf} x D={Df}: K2 + {nf} Adam steps + next step's K1/K1b in one pass")
    del buf2
    Of = torch.empty_like(Xf)
    param = torch.nn.Parameter(Xf[0])
    base = torch.optim.SGD([param], **sgd_kw)

    def unfused():
        ops.svgd_apply(Xf, Gf, Of, scf)
        for i in range(nf):     # svgd.py:92-103 with a single flat parameter (the best case for torch.optim)
            param.data = Xf[i]
            param.grad = Of[i]
            base.step()

    ms_unfused = time_kernel(unfused, 5, 2)
    ms_fused = res["svgd_apply_fused_sgd"]["ms"]
    res["svgd_apply_plus_base_optimizer"] = {
        "fused_ms": ms_fused, "k2_plus_torch_optim_ms": ms_unfused, "speedup": ms_unfused / ms_fused,
        "config": f"n={nf} x D={Df}, SGD momentum 0.9 nesterov wd 3e-4; unfused = bde K2 + {nf} x torch.optim.SGD.step() (foreach) on the same GPU"}
    log(f"[bench] K2 + base optimizer: fused {ms_fused:.3f} ms vs K2 + {nf} x torch.optim.SGD.step() {ms_unfused:.3f} ms "
        f"({ms_unfused / ms_fused:.2f}x)")
    del Xf, Gf, Of, buf, olast, param, base
    torch.cuda.empty_cache()
    # n = 20 (the CIFAR particle count) and n = 16 at a bandwidth-bound D: K1 = centred-Gram kernel, K2 on tensor-map tiles
    for nn_, Dn in ((20, 50_000_000), (16, 60_000_000)):
        Xn = torch.empty(nn_, Dn, device=dev)
        Gn = torch.empty(nn_, Dn, device=dev)
        for i in range(nn_):
            Xn[i].normal_(0.0, 0.05 * (1 + 0.1 * i), generator=g)
            Gn[i].normal_(0.0, 1e-3, generator=g)
        On = torch.empty_like(Xn)
        scn = ops.SvgdScratch.allocate(nn_, dev)
        rec(f"svgd_pairdist_n{nn_}", time_kernel(lambda: ops.svgd_pairdist_bandwidth(Xn, scn, L2_REG, KERNEL_GRAD_SCALE, DATASET_SIZE), 10, 3),
            4 * nn_ * Dn, f"n={nn_} x D={Dn}: K1 (centred Gram, tensor-map TMA) + fused K1b; exact redo fired: {scn.exact_redo()}")
        rec(f"svgd_apply_n{nn_}", time_kernel(lambda: ops.svgd_apply(Xn, Gn, On, scn), 10, 3), 12 * nn_ * Dn, f"n={nn_} x D={Dn}: K2")
        rec(f"svgd_step_n{nn_}", time_kernel(lambda: ops.svgd_step(Xn, Gn, On, scn, L2_REG, KERNEL_GRAD_SCALE, DATASET_SIZE), 10, 3),
            16 * nn_ * Dn, f"n={nn_} x D={Dn}: K1 + K1b + K2 (two launches + the conditional exact-redo launch)")
        bufn = torch.zeros(Dn, device=dev)
        rec(f"svgd_apply_fused_sgd_n{nn_}",
            time_kernel(lambda: ops.svgd_apply_sgd(Xn, Gn, scn, bufn, buf_initialized=True, lr=1e-7, momentum=0.9, nesterov=True,
                                                   weight_decay=3e-4), 10, 3),
            (12 * nn_ + 8) * Dn, f"n={nn_} x D={Dn}: K2 + {nn_} SGD steps in one pass, X in place")
        del Xn, Gn, On, scn, bufn
        torch.cuda.empty_cache()
    # C2 CIFAR ResNet-20 SVGD, n = 20 (small D: latency-bound, reported as time)
    n2, D2 = 20, 273_610
    D2p = (D2 + 63) // 64 * 64
    X2 = torch.randn(n2, D2p, device=dev, generator=g) * 0.05
    G2 = torch.randn(n2, D2p, device=dev, generator=g) * 1e-3
    O2 = torch.empty_like(X2)
    sc2 = ops.SvgdScratch.allocate(n2, dev)
    rec("svgd_step_n20_resnet20", time_kernel(lambda: ops.svgd_step(X2, G2, O2, sc2, 3e-4, 1.0, 50000.0), 20, 3, flush),
        16 * n2 * D2p, f"ResNet-20 D={D2}, n={n2} (FFMA-heavy, small D)")
    # C1 UCI MLP SVGD, n = 10, D = 501 (pure launch latency)
    X1 = torch.randn(10, 512, device=dev, generator=g)
    G1 = torch.randn(10, 512, device=dev, generator=g)
    O1 = torch.empty_like(X1)
    sc1 = ops.SvgdScratch.allocate(10, dev)
    rec("svgd_step_n10_uci", time_kernel(lambda: ops.svgd_step(X1, G1, O1, sc1, 0.01, 1.0, 768.0), 50, 5),
        16 * 10 * 512, "UCI MLP D=501, n=10 (launch latency)")
    return res


def k2_traffic(n, D):
    """DRAM bytes of one K2 launch from the committed ncu capture of this kernel (profiles/r02_k2_traffic.json:
    dram__bytes_read.sum + dram__bytes_write.sum at n = 10, D = 1e8), scaled to D; None for another n or without the file."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_k2_traffic.json")) as f:
            cap = json.load(f)
        if n != cap["n"]:
            return None
        return (cap["dram__bytes_read.sum"] + cap["dram__bytes_write.sum"]) * (D / cap["D"])
    except Exception:  # noqa: BLE001
        return None


def whole_step_configs(dev):
    """Whole `optimizer.step(forward_closure, backward_closure)` of the drop-in classes with REAL model closures at the
    small BASELINE configs (SURVEY §8d item ii: C1 = UCI MLP, SVGD n = 10, Adam; C2 = CIFAR ResNet-20-FRN, SVGD n = 20,
    SGD-Nesterov): wall clock per step, the model's forward + backward passes alone, and the difference — what the posterior
    update costs on top of the model, host-side Python included.  tests/perf_whole_step.py with kinds = ("b200",): only
    this package's classes run.  BDE_BENCH_WHOLE_STEP=C1,C2,C3,C4a,C4b widens it (C3 needs torchvision, C4 transformers)."""
    configs = [c for c in os.environ.get("BDE_BENCH_WHOLE_STEP", "C1,C2").split(",") if c]
    if not configs:
        return None
    try:
        tests_dir = os.path.join(ROOT, "tests")
        if tests_dir not in sys.path:
            sys.path.insert(0, tests_dir)
        import perf_whole_step
        res = perf_whole_step.run(configs, steps=3, warmup=2, kinds=("b200",), dev=dev)
        torch.cuda.empty_cache()
        log(f"[bench] whole step with model closures: { {k: v for k, v in res.items() if k != '_meta'} }")
        return res
    except Exception as e:  # noqa: BLE001
        log(f"[bench] whole-step configs failed: {e}")
        return {"error": str(e)}


def sharded_elementwise(ops, bdist, dist, world, rank, dev, iters=10):
    """N > 1: the elementwise family D-sharded (SURVEY §8e, second bullet) — every rank holds one slice of the SWAG and iVON
    state at the C3 / C4b sizes (weak: the slice IS a whole ResNet-50 / DistilBERT vector), placed in the job-wide Philox
    stream by dist.column_shard (the collective the host classes run at construction).  No data-path collective; timed like
    the headline step (barrier, CUDA events, max over ranks), aggregate = N x bytes / time."""
    res = {}

    def timed(fn, nbytes, name, cfg):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / iters], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        res[name] = {"ms": t.item(), "GBps_aggregate": world * nbytes / (t.item() * 1e-3) / 1e9, "config": cfg}

    g = torch.Generator(device=dev).manual_seed(11 + rank)
    D, K = 23_880_960, 10
    shard = bdist.column_shard(D, dist.group.WORLD)
    theta = torch.randn(D, device=dev, generator=g) * 0.05
    mean = theta + torch.randn(D, device=dev, generator=g) * 0.01
    sq = mean * mean + 1e-4
    ring = torch.randn(K, D, device=dev, generator=g) * 0.01
    out = torch.empty(D, device=dev)
    u = [0]

    def upd():
        u[0] += 1
        ops.swag_update(theta, mean, sq, ring[(u[0] - 1) % K], u[0])

    cfg = f"slice D={D} per GPU at elem0 = rank x D of {shard.total}, K={K}"
    timed(upd, 24 * D, "swag_update", cfg)
    timed(lambda: ops.swag_sample(mean, sq, ring, 3, out, seed=shard.seed, stream_id=2, elem0=shard.elem0), 4 * (K + 3) * D,
          "swag_sample", cfg)
    del theta, mean, sq, ring, out
    D = 66_955_072
    shard = bdist.column_shard(D, dist.group.WORLD)
    mean = torch.randn(D, device=dev, generator=g) * 0.05
    prec = torch.rand(D, device=dev, generator=g) * 1e-4 + 10.0 / 269038
    mom = torch.randn(D, device=dev, generator=g) * 1e-4
    dsum = torch.randn(D, device=dev, generator=g) * 0.3
    acc = torch.randn(D, device=dev, generator=g) * 2e-5
    theta = torch.zeros(D, device=dev)
    cfg = f"slice D={D} per GPU at elem0 = rank x D of {shard.total}"
    timed(lambda: ops.ivon_sample(mean, prec, dsum, theta, first=False, seed=shard.seed, stream_id=3, n_eff=269038.0,
                                  elem0=shard.elem0), 20 * D, "ivon_sample", cfg)
    dsum.normal_(0.0, 0.3, generator=g)
    step = [0]

    def ivon_upd():
        step[0] += 1
        ops.ivon_update(acc, dsum, mean, mom, prec, mc_samples=2, step=100 + step[0], lr=1e-5, beta1=0.9, beta2=0.999,
                        prior_prec=10.0, n_eff=269038.0, tempering=1.0, damping=1e-3)

    timed(ivon_upd, 32 * D, "ivon_update", cfg)
    res["elem0_of_this_rank"] = shard.elem0
    res["what"] = ("elementwise family D-sharded over the ranks: no collective on the data path; the group only places each "
                   "slice in the Philox stream (dist.column_shard)")
    del mean, prec, mom, dsum, acc, theta
    torch.cuda.empty_cache()
    if rank == 0:
        log(f"[bench] sharded elementwise family: {res}")
    return res


def sharded_closure(bde, dist, world, rank, dev, D=23_880_960, K=10, iters=10):
    """N > 1: a whole optimizer step on D-sharded state with a MODEL-shaped closure (SURVEY §8e last note, §8 f4):
    `ColumnShardedModel` all-gathers the ranks' weight slices before the forward and reduce-scatters the gradients after the
    backward (two single-buffer NCCL collectives over NVLink), `SwagOptimizer(process_group=...)` over a sharded SGD then
    updates 1 / N of the columns.  The model itself is left out (forward = a constant, backward = one accumulate pass into
    the pre-bound gradient views), so the lines show what sharding costs (the collectives) and saves (the update on 1 / N
    of the state) at ResNet-50 size; the unsharded class runs the same closure on every rank for comparison.  Strong
    scaling of a fixed D; barrier, CUDA events, max over ranks."""
    res = {}

    def timed(fn, name):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / iters], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        res[name] = {"ms": t.item()}
        return t.item()

    def make(group):
        g = torch.Generator(device=dev).manual_seed(5)
        w = torch.nn.Parameter(torch.randn(D, device=dev, generator=g) * 0.05)
        gsyn = torch.randn(D, device=dev, generator=g) * 1e-3
        zero = torch.zeros((), device=dev)
        sm = bde.ColumnShardedModel([w], group) if group is not None else None
        params = [sm.param] if sm is not None else [w]
        base = torch.optim.SGD(params, lr=0.01, momentum=0.9)
        opt = bde.SwagOptimizer(params, base, update_interval=1, deviation_samples=K, process_group=group)

        def fwd():
            return zero

        def bwd(loss):
            if w.grad is None:
                w.grad = gsyn.clone()
            else:
                w.grad.add_(gsyn)          # what autograd's AccumulateGrad does with a bound .grad
        return w, sm, opt, (sm.closures(fwd, bwd) if sm is not None else (fwd, bwd))

    w, sm, opt, (fwd, bwd) = make(dist.group.WORLD)
    wire = 4.0 * sm.shard * (world - 1)     # bytes every GPU receives (all-gather) / sends (reduce-scatter) per call
    ms = timed(sm.gather, "all_gather_weights")
    res["all_gather_weights"].update(GBps_per_gpu_on_the_wire=wire / (ms * 1e-3) / 1e9)
    ms = timed(sm.reduce_grads, "reduce_scatter_grads")
    res["reduce_scatter_grads"].update(GBps_per_gpu_on_the_wire=wire / (ms * 1e-3) / 1e9)
    timed(lambda: opt.step(fwd, bwd), "swag_step_sharded")
    res["swag_step_sharded"]["what"] = "gather + closure + reduce-scatter + SGD(momentum) and SWAG update on this rank's columns"
    res["state_bytes_per_gpu_sharded"] = 4 * sm.shard * (K + 4 + 1) + 8 * world * sm.shard
    shard_cols = sm.shard
    del w, sm, opt, fwd, bwd
    torch.cuda.empty_cache()
    w, _, opt, (fwd, bwd) = make(None)
    timed(lambda: opt.step(fwd, bwd), "swag_step_unsharded")
    res["swag_step_unsharded"]["what"] = "the plain class on the whole vector (every rank its own copy), same closure"
    res["state_bytes_per_gpu_unsharded"] = 4 * D * (K + 4 + 1) + 4 * D
    res["config"] = (f"flat weight vector D={D} (ResNet-50 size), K={K} deviations, {world} ranks x {shard_cols} columns; "
                     "model forward / backward left out")
    del w, opt, fwd, bwd
    torch.cuda.empty_cache()
    if rank == 0:
        log(f"[bench] sharded closure: {res}")
    return res


def strong_scaling(ops, bdist, dist, sc, n, world, rank, dev, in_kernel, steps):
    """D_total = 1e8 and 1e9 columns x n particles split over the `world` ranks (every rank [n, D_total / world]),
    timed like the headline step (barrier, CUDA events, max over ranks); rank 0 then runs the SAME total problem alone
    on its GPU, so the speed-up is measured inside one run.  With the in-kernel exchange the per-rank wait of K1's
    tail for its slowest peer (rank skew) is reported next to it."""
    from beyond_deep_ensembles_b200.layout import shard_bounds
    res = {}
    for D_total in (100_000_000, 1_000_000_000):
        lo, hi = shard_bounds(D_total, world, rank)
        Dl = hi - lo
        g = torch.Generator(device=dev).manual_seed(77 + rank)
        Xs = torch.empty(n, Dl, device=dev)
        Gs = torch.empty(n, Dl, device=dev)
        for i in range(n):
            Xs[i].normal_(0.0, 0.05 * (1 + 0.1 * i), generator=g)
            Gs[i].normal_(0.0, 1e-3, generator=g)
        Os = torch.empty_like(Xs)

        def one(scr, X_, G_, O_, single):
            if single or in_kernel:
                ops.svgd_pairdist_bandwidth(X_, scr, L2_REG, KERNEL_GRAD_SCALE, DATASET_SIZE)
            else:
                ops.svgd_pairdist(X_, scr)
                bdist.allreduce_dist(scr)
                ops.svgd_bandwidth(scr, L2_REG, KERNEL_GRAD_SCALE, DATASET_SIZE)
            ops.svgd_chain_next(X_)
            ops.svgd_apply(X_, G_, O_, scr)

        for _ in range(3):
            one(sc, Xs, Gs, Os, False)
        torch.cuda.synchronize()
        if sc.peers is not None:
            sc.peers.wait_stats(reset=True)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            one(sc, Xs, Gs, Os, False)
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        entry = {"D_total": D_total, "D_per_gpu": D_total // world, "ms_per_step": t.item(),
                 "GBps_aggregate": 16.0 * n * D_total / (t.item() * 1e-3) / 1e9}
        if sc.peers is not None:
            cnt, wsum, wmax = sc.peers.wait_stats(reset=True)
            w = torch.tensor([wsum / max(cnt, 1) / 1e3, wmax / 1e3], dtype=torch.float64, device=dev)
            allw = [torch.zeros_like(w) for _ in range(world)]
            dist.all_gather(allw, w)
            entry["peer_wait_us_per_rank"] = {"mean": [round(float(x[0]), 2) for x in allw],
                                              "max": [round(float(x[1]), 2) for x in allw],
                                              "what": "time K1's last CTA waited for its slowest peer per exchange (rank skew)"}
        del Xs, Gs, Os
        torch.cuda.empty_cache()
        if world > 1:
            t1 = torch.zeros(1, dtype=torch.float64, device=dev)
            if rank == 0:   # the same TOTAL problem on one GPU, unattached scratch
                sc1 = ops.SvgdScratch.allocate(n, dev)
                X1 = torch.empty(n, D_total, device=dev)
                G1 = torch.empty(n, D_total, device=dev)
                for i in range(n):
                    X1[i].normal_(0.0, 0.05 * (1 + 0.1 * i), generator=g)
                    G1[i].normal_(0.0, 1e-3, generator=g)
                O1 = torch.empty_like(X1)
                for _ in range(2):
                    one(sc1, X1, G1, O1, True)
                torch.cuda.synchronize()
                k = max(2, steps // 2)
                e0.record()
                for _ in range(k):
                    one(sc1, X1, G1, O1, True)
                e1.record()
                torch.cuda.synchronize()
                t1[0] = e0.elapsed_time(e1) / k
                del X1, G1, O1, sc1
                torch.cuda.empty_cache()
            dist.all_reduce(t1, op=dist.ReduceOp.MAX)
            entry["ms_per_step_1gpu_same_total"] = t1.item()
            entry["speedup"] = t1.item() / t.item()
            entry["efficiency"] = t1.item() / t.item() / world
        res[f"D{D_total:.0e}".replace("+0", "").replace("+", "")] = entry
        if rank == 0:
            log(f"[bench] strong D_total={D_total}: {entry}")
    return res


def make_inputs(n, D, rank, dev):
    """Synthetic, device-resident inputs of the timed step: particles X and gradients G [n, D] of this rank's column
    slice [rank*D, (rank+1)*D), seeded by the rank, so every run with the same arguments gets the same ones."""
    g = torch.Generator(device=dev).manual_seed(1000 + rank)
    X = torch.randn(n, D, device=dev, generator=g)
    X *= (0.05 * (1 + 0.1 * torch.arange(n, device=dev, dtype=torch.float32))).unsqueeze(1)
    G = torch.randn(n, D, device=dev, generator=g) * 1e-3
    return X, G


def dump_outputs(path, out, sc, world, rank):
    """--dump-outputs: what a caller of the timed step holds after its last step, as .npy files in `path`.
    out.npy: the update direction [n, D] of this rank's columns, float32, at DUMP_COLUMNS // world columns drawn
    without replacement by a fixed seed and kept in column order (every column when D is smaller); with N > 1 each
    rank writes out_rank<r>.npy.  pair_dist, kernel_K, kernel_A, bandwidth_info (h, median, d_lo, d_hi) and
    median_sel: the scratch the step leaves, the same on every rank, written by rank 0 (float64; K and A float32).
    The inputs are seeded, so two builds run with the same arguments can be compared file for file."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    D = out.shape[1]
    cols = DUMP_COLUMNS // world
    if D > cols:
        idx = np.sort(np.random.default_rng(0).choice(D, cols, replace=False))
        out = out[:, torch.from_numpy(idx).to(out.device)]
    np.save(os.path.join(path, "out.npy" if world == 1 else f"out_rank{rank}.npy"), out.cpu().numpy())
    if rank == 0:
        for name, t in (("pair_dist", sc.dist), ("kernel_K", sc.K), ("kernel_A", sc.A), ("bandwidth_info", sc.info),
                        ("median_sel", sc.sel.double())):
            np.save(os.path.join(path, f"{name}.npy"), t.cpu().numpy())


# --------------------------------------------------------------------------------------
def main():
    global D_PER_GPU
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of the headline workload")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--d-per-gpu", type=int, default=D_PER_GPU, help=argparse.SUPPRESS)
    ap.add_argument("--skip-extras", action="store_true", help="skip e2e / cpu baseline / other paths (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")

    if args.impl == "reference":
        run_reference_arm(args)
        return

    # stdout carries exactly ONE JSON line: everything else that might print there (NCCL's version banner,
    # library chatter) is sent to stderr by re-pointing fd 1; the line itself goes to the saved descriptor
    json_fd = os.dup(1)
    os.dup2(2, 1)

    D_PER_GPU = args.d_per_gpu
    import torch.distributed as dist
    from beyond_deep_ensembles_b200 import _lib, ops
    from beyond_deep_ensembles_b200 import dist as bdist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        log(f"[bench] WORLD_SIZE={world} but --gpus {args.gpus}: launch with torch.distributed.run for N > 1")
        if world == 1 and args.gpus > 1:
            raise SystemExit(2)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    _lib.get()  # fail loudly if libbde_b200.so is missing
    peak_gbs, peak_src = measured_peaks()
    warmup = max(3, args.warmup)
    steps = args.steps
    n, D = N_PARTICLES, D_PER_GPU

    X, G = make_inputs(n, D, rank, dev)
    out = torch.empty_like(X)
    sc = ops.SvgdScratch.allocate(n, dev)

    # N > 1: the n*n partial distances are summed across ranks inside K1's tail over peer memory (CUDA IPC +
    # NVLink) when the ranks can map each other; otherwise K1 -> NCCL all-reduce -> K1b
    peer = world > 1 and bdist.enable_peer_exchange(sc)
    in_kernel = [world == 1 or peer]

    def step(events=None):
        """One posterior update; `events` collects (K1 start, K1 end / K2 start, K2 end)."""
        if events is not None:
            events[0].record()
        if in_kernel[0]:
            ops.svgd_pairdist_bandwidth(X, sc, L2_REG, KERNEL_GRAD_SCALE, DATASET_SIZE)
        else:
            ops.svgd_pairdist(X, sc)
            bdist.allreduce_dist(sc)
            ops.svgd_bandwidth(sc, L2_REG, KERNEL_GRAD_SCALE, DATASET_SIZE)
        if events is not None:
            events[1].record()
        # K2 is launched as a programmatic dependent of K1 (its ring fills during K1's tail); the event between the two
        # is a marker on the stream and takes its timestamp when K1 completes
        ops.svgd_chain_next(X)
        ops.svgd_apply(X, G, out, sc)
        if events is not None:
            events[2].record()

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()

    launches0 = _lib.launch_count
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
    t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # the sampler thread (NVML init) starts BEFORE the barrier: anything rank-variable between the barrier and
    # t_begin shows up as start skew, which the in-kernel exchange of step 1 would charge to the fastest rank
    with ClockSampler(local_rank) as clocks:
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t_begin.record()
        for s in range(steps):
            step(evs[s])
        t_end.record()
        torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches = _lib.launch_count - launches0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out, sc, world, rank)

    total_ms = t_begin.elapsed_time(t_end)
    k1_ms = sum(e[0].elapsed_time(e[1]) for e in evs) / steps
    k2_ms = sum(e[1].elapsed_time(e[2]) for e in evs) / steps
    tm = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    total_ms = tm.item()
    ms_per_step = total_ms / steps
    value = 16.0 * n * D * world / (ms_per_step * 1e-3) / 1e9

    # N > 1 with the peer exchange: also time the portable form (K1 -> NCCL all-reduce -> K1b -> K2) for comparison
    exchange = None
    if world > 1:
        exchange = {"form": "in-kernel peer exchange (P2P stores + epoch flags in K1's tail)" if peer else
                    "NCCL all-reduce of n*n fp64 between K1 and K1b", "launches_per_step": 2 if peer else 4}
        if peer:
            sc_nccl = ops.SvgdScratch.allocate(n, dev)
            sc_peer, sc = sc, sc_nccl
            in_kernel[0] = False
            for _ in range(warmup):
                step()
            torch.cuda.synchronize()
            dist.barrier()
            torch.cuda.synchronize()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(steps):
                step()
            a1.record()
            torch.cuda.synchronize()
            tn = torch.tensor([a0.elapsed_time(a1)], dtype=torch.float64, device=dev)
            dist.all_reduce(tn, op=dist.ReduceOp.MAX)
            exchange["nccl_form_ms_per_step"] = tn.item() / steps
            exchange["peer_form_ms_per_step"] = ms_per_step
            same = torch.equal(sc_nccl.sel, sc_peer.sel) and torch.allclose(sc_nccl.dist, sc_peer.dist, rtol=1e-12, atol=0)
            exchange["peer_equals_nccl"] = bool(same)
            exchange["peer_status_epochs_timeouts"] = list(sc_peer.peers.status())
            sc = sc_peer
            in_kernel[0] = True

    # ---- strong scaling: a FIXED total problem split N ways (north star: near-linear 1 -> 8 at D >= 100 M x 10) ----
    strong = None
    if not args.skip_extras:
        del out
        strong = strong_scaling(ops, bdist, dist, sc, n, world, rank, dev, in_kernel[0], max(3, min(steps, 10)))
        out = torch.empty_like(X)
        step()   # K / A of the headline problem back in the scratch, `out` refilled (the e2e leg compares against it)

    sharded_ew = None
    if world > 1 and not args.skip_extras:
        try:
            sharded_ew = sharded_elementwise(ops, bdist, dist, world, rank, dev)
        except Exception as e:  # noqa: BLE001
            log(f"[bench] sharded elementwise family failed: {e}")
            sharded_ew = {"error": str(e)}

    sharded_cl = None
    if world > 1 and not args.skip_extras:
        try:
            import beyond_deep_ensembles_b200 as bde
            sharded_cl = sharded_closure(bde, dist, world, rank, dev)
        except Exception as e:  # noqa: BLE001
            log(f"[bench] sharded closure failed: {e}")
            sharded_cl = {"error": str(e)}

    # ---- end-to-end through the host-buffer API (pinned host memory, H2D + D2H inside the timing) ----
    e2e = {"value": None, "unit": "GB/s", "h2d_bytes_per_step": 8 * n * D * world, "d2h_bytes_per_step": 4 * n * D * world}
    paths, cpu_base, eager, whole = None, None, None, None
    if not args.skip_extras:
        try:
            import psutil
            need = 3 * 4 * n * D * world
            avail = psutil.virtual_memory().available
            if avail < 2 * need:
                raise RuntimeError(f"host memory: need {need >> 30} GiB pinned, {avail >> 30} GiB available")
            Xh = torch.empty((n, D), dtype=torch.float32, pin_memory=True)
            Gh = torch.empty((n, D), dtype=torch.float32, pin_memory=True)
            Oh = torch.empty((n, D), dtype=torch.float32, pin_memory=True)
            Xh.copy_(X)
            Gh.copy_(G)
            ref_cols = out[:, :1024].cpu()
            del out
            torch.cuda.empty_cache()
            st = ops.HostStaging.allocate(n, D, 4_000_000, dev, dX=X if D % 4 == 0 else None)
            e2e_steps = min(steps, 5)
            sc_host = ops.SvgdScratch.allocate(n, dev) if sc.peers is not None else sc   # host path: all-reduce form

            def e2e_step():
                ops.svgd_step_host(Xh, Gh, Oh, st, sc_host, L2_REG, KERNEL_GRAD_SCALE, DATASET_SIZE)

            e2e_step()  # warm-up (page-locks, stream creation)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                e2e_step()
            torch.cuda.synchronize()
            dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            e2e_ms = 1e3 * dt.item() / e2e_steps
            if not torch.allclose(Oh[:, :1024], ref_cols, rtol=1e-5, atol=1e-6):
                raise RuntimeError("end-to-end result differs from the device-resident step")
            e2e.update(value=16.0 * n * D * world / (e2e_ms * 1e-3) / 1e9, ms_per_step=e2e_ms, steps=e2e_steps,
                       api="ops.svgd_step_host -> bde_svgd_host_pairdist / bde_svgd_host_apply (C-ABI, pinned host buffers)")
            del Xh, Gh, Oh, st
        except Exception as e:  # noqa: BLE001
            log(f"[bench] e2e skipped: {e}")
            e2e["skipped"] = str(e)

        if rank == 0 and world == 1:
            del X, G
            torch.cuda.empty_cache()
            try:
                paths = other_paths(ops, peak_gbs, dev)
            except Exception as e:  # noqa: BLE001
                log(f"[bench] other paths failed: {e}")
                paths = {"error": str(e)}
            whole = whole_step_configs(dev)
            eager = eager_cuda_reference(dev)
            gbs, ms, threads, kind, Dc = cpu_reference_run(3, 1)
            cpu_base = {"value": gbs, "unit": "GB/s", "ms_per_step": ms, "cores": threads, "kind": kind,
                        "sample": cpu_sample_text(kind, Dc, 3) + ", all host threads"}
            gbs8, ms8, t8, _, _ = cpu_reference_run(2, 1, threads=min(8, os.cpu_count() or 1))   # SURVEY §8d: second run pinned to 8 threads
            cpu_base["pinned_threads_run"] = {"value": gbs8, "unit": "GB/s", "ms_per_step": ms8, "cores": t8}

    if rank == 0:
        k2_bytes = 12.0 * n * D
        k1_bytes = 4.0 * n * D
        k2_gbs = k2_bytes / (k2_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(world),
            "clocks": clocks.summary(), "e2e": e2e, "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": "bde::svgd_apply_tma_kernel<10, 0, false, 3, 256> (K2: out = K G + A X; 3 tile sets x 256 columns)",
                         "achieved": k2_gbs, "peak": peak_gbs, "unit": "GB/s", "frac": k2_gbs / peak_gbs,
                         "peak_source": peak_src, "frac_of_nominal_8TBps": k2_gbs / 8000.0,
                         "algorithmic_bytes_per_launch": k2_bytes, "ms_per_launch": k2_ms,
                         # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of this kernel
                         # at n=10, D=1e8 (profiles/r02_ncu_summary.md, tensor-map kernel): 8.000 GB + 3.970 GB per launch.
                         # A citation of that capture, not a live counter: ncu cannot run inside the timed region.
                         "traffic": k2_traffic(n, D),
                         "traffic_source": "profiles/r02_k2_traffic.json (ncu --set full capture r02_prof_n10.ncu-rep, "
                                           "tools/sessions/r02_s11.sh; read in profiles/r02_ncu_summary.md)"},
            "kernels": {
                "svgd_pairdist(+bandwidth)": {"ms": k1_ms, "GBps": k1_bytes / (k1_ms * 1e-3) / 1e9,
                                               "frac": k1_bytes / (k1_ms * 1e-3) / 1e9 / peak_gbs,
                                               "algorithmic_bytes": k1_bytes,
                                               "includes": ("in-kernel peer exchange + fused K1b tail" if peer else
                                                            "n*n all-reduce + K1b") if world > 1 else "fused K1b tail"},
                "svgd_apply": {"ms": k2_ms, "GBps": k2_gbs, "frac": k2_gbs / peak_gbs, "algorithmic_bytes": k2_bytes},
            },
            "step_frac_of_measured_peak": value / world / peak_gbs,
            "step_frac_of_nominal_8TBps": value / world / 8000.0,
            "cpu_baseline": cpu_base, "eager_cuda": eager, "paths": paths, "exchange": exchange, "strong": strong, "sharded_elementwise": sharded_ew, "sharded_closure": sharded_cl,
            "whole_step": whole,
        }
        os.write(json_fd, (json.dumps(line) + "\n").encode())
        try:
            os.fsync(json_fd)
        except OSError:
            pass
    if world > 1:
        dist.barrier()
        bdist.shutdown_peer_exchange()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

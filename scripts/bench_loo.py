#!/usr/bin/env python
"""Model comparison on one GPU: the pointwise log-likelihood matrix (k_ll_obs / k_ll_custom_obs) and the PSIS step
(k_psis) of demcmc_loo at S = 4000 draws and N = 1e5 observations:

  gaussian   Normal(mu, sigma), 1e5 observations
  lba        LBA, 2 accumulators, 1e5 trials (the configs[2] data of scripts/bench_configs.py)
  mvnormal   isotropic MVN d = 50, 1e5 observations (the configs[1] data)
  custom_lba the same LBA written as a DEMCMC_CUSTOM source (scripts/bench_custom.py), compiled at run time

The draws are spread around the parameters that generated the data.  Per workload, after one warm-up call of the same
shape: the host time of demcmc_loo (it ends in the download of the four outputs; median of --reps calls, profiler off),
then, in a separate profiled call (torch.profiler, CUDA activities), the device time of every kernel of demcmc_loo: the
pointwise kernels (k_ll_obs_prep + k_ll_obs, or k_ll_custom_obs) give the densities per second, k_psis the cost of the
PSIS step (what demcmc_loo costs beyond demcmc_eval_pointwise's kernels; the host time of demcmc_eval_pointwise itself is
dominated by handing 3.2 GB to the host and is not what the step costs).  For mvnormal the share of the fp64 peak
(demcmc_fp64_peak, measured in the same run) counts 3 flops per (observation, dimension, draw).  The first line names
the card and its power limit (nvidia-smi, read only).

Usage: python scripts/bench_loo.py [--out profiles/loo_bench.jsonl] [--reps 5] [workload ...]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import demcmc_b200 as D  # noqa: E402
from bench_configs import config  # noqa: E402
from bench_custom import LBA as LBA_SOURCE  # noqa: E402

S, N = 4000, 100_000


def workload(name, rng):
    """(set_model kwargs, d, draws[S][d], the name of the pointwise kernels)"""
    if name == "gaussian":
        x = rng.normal(0.3, 1.2, N)
        return dict(kind="gaussian", x=x), 2, np.column_stack([rng.normal(0.3, 0.004, S), rng.normal(1.2, 0.003, S)]), "k_ll_obs"
    if name in ("lba", "custom_lba"):
        c = config("c3")
        rt, choice = c["data"]["x"], c["data"]["choice"]
        th = np.column_stack([rng.normal([3, 2], 0.01, (S, 2)), rng.normal(0.8, 0.003, S), rng.normal(0.2, 0.002, S),
                              rng.uniform(0.295, 0.3, S)])
        if name == "lba":
            return dict(kind="lba", x=rt, choice=choice, n_dim=2), 5, th, "k_ll_obs"
        return dict(kind="custom", x=np.column_stack([rt, choice.astype(float)]), source=LBA_SOURCE), 5, th, "k_ll_custom_obs"
    if name == "mvnormal":
        c = config("c2")
        x = c["data"]["x"]
        mu = x.mean(axis=0)
        th = np.column_stack([rng.normal(mu, 0.003, (S, mu.size)), rng.normal(1.0, 0.002, S)])
        return dict(kind="mvnormal", x=x), mu.size + 1, th, "k_ll_obs"
    raise KeyError(name)


def kernel_times(h, th):
    """device time (ms) per kernel name of one demcmc_loo call, from torch.profiler's CUDA activities"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        h.loo(th)
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            out[e.key] = out.get(e.key, 0.0) + t / 1000.0
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "loo_bench.jsonl"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("workloads", nargs="*", default=["gaussian", "lba", "mvnormal", "custom_lba"])
    a = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    peak = D.fp64_peak(0)
    lines = [dict(what="device", nvidia_smi=smi, fp64_peak_tflops=peak, draws=S, observations=N)]
    print(json.dumps(lines[-1]), flush=True)
    rng = np.random.default_rng(4242)
    for name in a.workloads:
        kw, d, th, prefix = workload(name, rng)
        kind = kw.pop("kind")
        with D.Handle(1, 3, d, [-np.inf] * d, [np.inf] * d) as h:
            h.set_model(kind, [("flat",)] * d, **kw)
            h.loo(th)                                        # warm-up: module load, pool growth, the custom compile
            times = []
            for _ in range(a.reps):
                t0 = time.perf_counter()
                res = h.loo(th)
                times.append((time.perf_counter() - t0) * 1e3)
            kt = kernel_times(h, th)
        pw_ms = sum(v for k, v in kt.items() if prefix in k)          # (names are demangled signatures: "void de::be::k_ll_obs<0>(...)")
        psis_ms = sum(v for k, v in kt.items() if "k_psis" in k)
        if not (pw_ms > 0 and psis_ms > 0):
            raise RuntimeError(f"the profiler saw no pointwise / PSIS kernel: {kt}")
        rec = dict(what=name, draws=S, observations=N, loo_host_ms=float(np.median(times)), loo_host_ms_all=times,
                   pointwise_kernel_ms=pw_ms, psis_kernel_ms=psis_ms, kernels_ms=kt,
                   densities_per_s=S * N / (pw_ms * 1e-3), pareto_k_above_0_7=int(np.sum(res[1] > 0.7)),
                   elpd_loo=float(np.sum(res[0])))
        if name == "mvnormal":
            rec["fp64_tflops"] = 3.0 * S * N * (d - 1) / (pw_ms * 1e-3) / 1e12
            rec["fp64_peak_share"] = rec["fp64_tflops"] / peak
        lines.append(rec)
        print(json.dumps(rec), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for r in lines:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Custom (run-time compiled) likelihoods against the registered kernels of the same densities, one GPU.

For each workload the registered kind and a DEMCMC_CUSTOM source of the same density run alternately, `--rounds` times
each, on the same data, seed and initial states:

  gaussian   Normal(mu, sigma), 1e5 observations, 4 groups x 256 particles (burn-in: select_base on)
  lba        LBA, 2 accumulators, 1e5 trials, 4 x 256 (the configs[2] shape of scripts/bench_configs.py)
  lnr        LNR, 4 accumulators, 1e5 trials, 4 x 256
  gaussian_small  the reference's Gaussian_Example size: 50 observations, 4 x 6 (the registered kind runs the
                  single-CTA chunk kernel there; a custom model never does)

Per run: particle updates/s (CUDA events around the whole run call, demcmc_counters.device_ms), the device time of the
likelihood kernel per iteration from a second, separately timed pass (demcmc_set_timing time_loglik: CUDA events around
every likelihood launch), and the wall time of demcmc_set_model -- for a custom source the first set_model of the
process includes the NVRTC compile, the later ones hit the cache.  The first line names the card, its power limit and
its maximum SM clock (nvidia-smi, read only).  One JSON line per run, then one summary line per workload with the
medians and the custom / registered ratio.

Usage: python scripts/bench_custom.py [--rounds 3] [workload ...]
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
from bench_configs import lba_sim_vec  # noqa: E402

INF = np.inf
LOG2PI = "1.8378770664093454836"

GAUSS = """
#define DEMCMC_NPAR 3
__device__ void demcmc_prepare(const double *theta, double *par) { par[0] = theta[0]; par[1] = theta[1]; par[2] = log(theta[1]); }
__device__ double demcmc_obs(const double *par, const double *x)
{
    const double z = (x[0] - par[0]) / par[1];
    return -(z * z + LOG2PI) / 2.0 - par[2];
}
""".replace("LOG2PI", LOG2PI)
LNR = """
__device__ double demcmc_obs(const double *par, const double *x)
{
    const double t = x[0] - par[4];
    if (!(t > 0.0)) return t != t ? DEMCMC_NAN : -DEMCMC_INF;
    const double lx = log(t);
    const int c = (int)x[1] - 1;
    double ll = 0.0;
    for (int r = 0; r < 4; ++r) {
        const double z = lx - par[r];
        if (r == c) ll += -(z * z + LOG2PI) / 2.0 - lx;
        else {
            const double u = z * 0.70710678118654752440;
            ll += u < 5.0 ? log(0.5 * erfc(u)) : log(0.5 * erfcx(u)) - u * u;
        }
    }
    return ll;
}
""".replace("LOG2PI", LOG2PI)
LBA = """
#define DEMCMC_NPAR 6
__device__ void demcmc_prepare(const double *th, double *par)
{
    double pneg = 1.0;
    for (int r = 0; r < 5; ++r) par[r] = th[r];
    for (int r = 0; r < 2; ++r) pneg *= 0.5 * erfc(th[r] * 0.70710678118654752440);
    par[5] = 1.0 / (1.0 - pneg);
}
__device__ double demcmc_obs(const double *par, const double *x)
{
    const double A = par[2], b = A + par[3], tau = par[4], rt = x[0];
    const int c = (int)x[1] - 1;
    if (rt < tau) return log(1e-10);
    const double dt = rt - tau;
    double den = 1.0;
    for (int r = 0; r < 2; ++r) {
        const double v = par[r];
        const double n1 = (b - A - dt * v) / dt, n2 = (b - dt * v) / dt;
        const double c1 = 0.5 * erfc(-n1 * 0.70710678118654752440), c2 = 0.5 * erfc(-n2 * 0.70710678118654752440);
        const double p1 = exp(-0.5 * n1 * n1) * 0.39894228040143267794, p2 = exp(-0.5 * n2 * n2) * 0.39894228040143267794;
        if (r == c) {
            const double f = (-v * c1 + p1 + v * c2 - p2) / A;
            den *= f > 0.0 ? f : (f != f ? f : 0.0);
        } else {
            double F = 1.0 + ((b - A - dt * v) / A) * c1 - ((b - dt * v) / A) * c2 + (dt / A) * p1 - (dt / A) * p2;
            F = F > 0.0 ? F : (F != F ? F : 0.0);
            den *= 1.0 - F;
        }
    }
    den *= par[5];
    if (den != den) return -DEMCMC_INF;
    return log(den < 1e-10 ? 1e-10 : den);
}
"""


def workload(name):
    """(registered set_model kwargs, custom set_model kwargs, G, Np, d, prior, lo, hi, theta0, iterations)"""
    if name in ("gaussian", "gaussian_small"):
        n, G, Np, iters = (100_000, 4, 256, 200) if name == "gaussian" else (50, 4, 6, 2000)
        x = np.random.default_rng(50514).normal(0.0, 1.0, n)
        return (dict(kind="gaussian", x=x), dict(kind="custom", x=x, source=GAUSS), G, Np, 2,
                [("normal", 0, 1), ("halfcauchy", 0, 1)], [-INF, 0.0], [INF, INF],
                lambda r, P: np.column_stack([r.normal(size=P), np.abs(r.standard_cauchy(P)) + 0.1]), iters)
    if name == "lba":
        choice, rt = lba_sim_vec(np.random.default_rng(88484), 100_000)
        mn = float(rt.min())
        prior = [("normal", 1, 5), ("normal", 1, 5), ("normal", 0.8, 0.2), ("normal", 0.2, 0.1), ("uniform", 0, mn)]
        return (dict(kind="lba", x=rt, choice=choice, n_dim=2), dict(kind="custom", x=np.column_stack([rt, choice.astype(float)]), source=LBA),
                4, 256, 5, prior, [0, 0, 0, 0, 0], [INF, INF, INF, INF, mn],
                lambda r, P: np.column_stack([np.abs(r.normal(1, 5, P)), np.abs(r.normal(1, 5, P)), np.abs(r.normal(0.8, 0.2, P)),
                                              np.abs(r.normal(0.2, 0.1, P)), r.uniform(0, mn, P)]), 60)
    if name == "lnr":
        rng = np.random.default_rng(4407)
        x = np.exp(rng.normal((-2.0, -2.0, -3.0, -3.0), 1.0, size=(100_000, 4)))
        choice, rt = (np.argmin(x, axis=1) + 1).astype(np.int32), 0.5 + x.min(axis=1)
        mn = float(rt.min())
        return (dict(kind="lnr", x=rt, choice=choice, n_dim=4), dict(kind="custom", x=np.column_stack([rt, choice.astype(float)]), source=LNR),
                4, 256, 5, [("normal", 0, 3)] * 4 + [("uniform", 0, mn)], [-INF] * 4 + [0.0], [INF] * 4 + [mn],
                lambda r, P: np.column_stack([r.normal(-2, 1, (P, 4)), r.uniform(0, mn, P)]), 60)
    raise KeyError(name)


def run(name, impl, wl):
    reg, cus, G, Np, d, prior, lo, hi, theta0, iters = wl
    model = dict(reg if impl == "registered" else cus)
    kind = model.pop("kind")
    h = D.Handle(G, Np, d, lo, hi, seed=20261017, burnin=iters // 2)
    try:
        t0 = time.perf_counter()
        h.set_model(kind, prior, **model)
        set_model_s = time.perf_counter() - t0
        h.set_state(theta0(np.random.default_rng(1), G * Np))
        h.run(max(3, iters // 10))                                  # warm-up: module load, allocations
        c0 = h.counters()
        h.run(iters)
        c1 = h.counters()
        h.set_timing(0, True)                                       # a separate pass: events around every likelihood launch
        h.run(iters)
        c2 = h.counters()
    finally:
        h.close()
    ups = (c1["particle_updates"] - c0["particle_updates"]) / (c1["device_ms"] * 1e-3)
    return {"workload": name, "impl": impl, "particles": G * Np, "iterations": iters, "particle_updates_per_s": ups,
            "ms_per_iteration": c1["device_ms"] / iters, "loglike_kernel_ms_per_iteration": c2["loglike_ms"] / iters,
            "kernel_launches_per_iteration": (c1["kernel_launches"] - c0["kernel_launches"]) / iters, "set_model_s": set_model_s}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("workloads", nargs="*", default=["gaussian", "lba", "lnr", "gaussian_small"])
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    D._ffi.use_library(D._ffi.DEFAULT_LIB)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    print(json.dumps({"nvidia_smi": smi.stdout.strip().splitlines()}), flush=True)
    for name in a.workloads:
        wl = workload(name)
        rows = {"registered": [], "custom": []}
        for _ in range(a.rounds):
            for impl in ("registered", "custom"):
                r = run(name, impl, wl)
                rows[impl].append(r)
                print(json.dumps(r), flush=True)
        med = {k: {m: float(np.median([r[m] for r in v])) for m in ("particle_updates_per_s", "loglike_kernel_ms_per_iteration")}
               for k, v in rows.items()}
        cs = [r["set_model_s"] for r in rows["custom"]]
        print(json.dumps({"workload": name, "summary": med,
                          "custom_over_registered_updates_per_s": med["custom"]["particle_updates_per_s"] / med["registered"]["particle_updates_per_s"],
                          "custom_over_registered_loglike_kernel_time": med["custom"]["loglike_kernel_ms_per_iteration"] / max(1e-12, med["registered"]["loglike_kernel_ms_per_iteration"]),
                          "custom_set_model_s_first": cs[0], "custom_set_model_s_cached": float(np.median(cs[1:])) if len(cs) > 1 else None}), flush=True)


if __name__ == "__main__":
    main()

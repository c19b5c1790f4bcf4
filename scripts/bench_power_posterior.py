#!/usr/bin/env python
"""Power posteriors on one GPU: K = 32 rungs in ONE handle (K x 4 groups, demcmc_set_temperatures) against one rung alone
(4 groups at t = 1), at the same particles per rung and the same iterations:

  lba       LBA, 2 accumulators, 500 trials, 4 x 24 per rung, 2000 iterations
  gaussian  Normal(mu, sigma), 50 observations, 4 x 6 per rung, 2000 iterations
  mvnormal  isotropic MVN d = 50, 1e5 observations (the configs[1] shape of scripts/bench_configs.py), 4 x 256 per rung,
            20 iterations

Per workload and layout, after a warm-up run of the same shape: the host time of demcmc_run (it ends in a device
synchronise) and of demcmc_power_posterior over every stored row (the K-rung handle only; one rung alone has no ladder),
median of --reps.  Reported: particle updates per second, the wall time to a log Z (run + evidence), and
ratio = time(K rungs) / (K * time(one rung)) as measured.  Then the time of one demcmc_power_posterior call at K = 32 and
2000 stored rows (the gaussian handle).  The first line names the card, its power limit and its max SM clock (nvidia-smi,
read only).

Usage: python scripts/bench_power_posterior.py [--out profiles/power_posterior_bench.jsonl] [--reps 3] [workload ...]
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
K = 32


def workload(name):
    rng = np.random.default_rng(2026)
    if name == "lba":
        choice, rt = lba_sim_vec(rng, 500)
        mn = float(rt.min())
        prior = [("normal", 1, 5), ("normal", 1, 5), ("normal", 0.8, 0.2), ("normal", 0.2, 0.1), ("uniform", 0, mn)]
        th0 = lambda r, P: np.column_stack([np.abs(r.normal(1, 5, P)), np.abs(r.normal(1, 5, P)), np.abs(r.normal(0.8, 0.2, P)),  # noqa: E731
                                            np.abs(r.normal(0.2, 0.1, P)), r.uniform(0, mn, P)])
        return dict(kind="lba", Np=24, d=5, prior=prior, lo=[0] * 5, hi=[INF] * 4 + [mn], data=dict(x=rt, choice=choice, n_dim=2),
                    theta0=th0, iters=2000)
    if name == "gaussian":
        x = rng.normal(0, 1, 50)
        return dict(kind="gaussian", Np=6, d=2, prior=[("normal", 0, 10), ("halfcauchy", 0, 1)], lo=[-INF, 0], hi=[INF, INF],
                    data=dict(x=x), theta0=lambda r, P: np.column_stack([r.normal(size=P), np.abs(r.standard_cauchy(P)) + 0.1]), iters=2000)
    if name == "mvnormal":
        dm = 50
        mu = rng.normal(size=dm)
        x = rng.normal(mu, 1.0, size=(100_000, dm))
        return dict(kind="mvnormal", Np=256, d=dm + 1, prior=[("normal", 0, 1)] * dm + [("halfcauchy", 0, 1)], lo=[-INF] * dm + [0.0],
                    hi=[INF] * (dm + 1), data=dict(x=x),
                    theta0=lambda r, P: np.column_stack([r.normal(size=(P, dm)), np.abs(r.standard_cauchy(P)) + 0.1]), iters=20)
    raise KeyError(name)


def timed(c, n_rungs, reps):
    G = 4 * n_rungs
    t = np.repeat((np.arange(n_rungs) / max(n_rungs - 1, 1)) ** 5 if n_rungs > 1 else np.ones(1), 4)
    runs, evid, out = [], [], None
    for rep in range(reps + 1):                       # rep 0: warm-up of the same shape
        with D.Handle(G, c["Np"], c["d"], c["lo"], c["hi"], alpha=0.0, burnin=0, seed=7 + rep) as h:
            h.set_model(c["kind"], c["prior"], **c["data"])
            h.set_temperatures(t)
            h.set_state(c["theta0"](np.random.default_rng(rep), G * c["Np"]))
            t0 = time.perf_counter()
            h.run(c["iters"])
            t1 = time.perf_counter()
            if n_rungs > 1:
                out = h.power_posterior(0, h.n_rows)
            t2 = time.perf_counter()
            if rep:
                runs.append(t1 - t0)
                evid.append(t2 - t1)
    run_s, ev_s = float(np.median(runs)), float(np.median(evid))
    ups = G * c["Np"] * c["iters"] / run_s
    res = dict(rungs=n_rungs, groups=G, Np=c["Np"], iterations=c["iters"], run_s=run_s, evidence_s=ev_s, updates_per_s=ups,
               wall_to_log_z_s=run_s + ev_s)
    if out is not None:
        res.update(log_z_ti=out["log_z_ti"], log_z_ti2=out["log_z_ti2"], log_z_ss=out["log_z_ss"], se_ti=out["se_ti"], se_ss=out["se_ss"])
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "power_posterior_bench.jsonl"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("workloads", nargs="*", default=["lba", "gaussian", "mvnormal"])
    a = ap.parse_args()
    D._ffi.use_library(D._ffi.DEFAULT_LIB)
    if D._ffi.lib().demcmc_backend_name() != b"cuda-sm100a" or D._ffi.lib().demcmc_device_count() < 1:
        raise SystemExit("needs the CUDA library and a GPU")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    lines = [dict(device=smi[0] if smi else "unknown")]
    for name in a.workloads:
        c = workload(name)
        many, one = timed(c, K, a.reps), timed(c, 1, a.reps)
        lines.append(dict(workload=name, k_rungs=many, one_rung=one, ratio=many["run_s"] / (K * one["run_s"])))
        print(json.dumps(lines[-1]), flush=True)
    # one demcmc_power_posterior call at K = 32 rungs and 2000 stored rows
    c = workload("gaussian")
    G = 4 * K
    with D.Handle(G, c["Np"], c["d"], c["lo"], c["hi"], alpha=0.0, burnin=0, seed=3) as h:
        h.set_model(c["kind"], c["prior"], **c["data"])
        h.set_temperatures(np.repeat((np.arange(K) / (K - 1)) ** 5, 4))
        h.set_state(c["theta0"](np.random.default_rng(0), G * c["Np"]))
        h.run(2000)
        h.power_posterior(0, 2000)
        ts = []
        for _ in range(10):
            t0 = time.perf_counter()
            h.power_posterior(0, 2000)
            ts.append(time.perf_counter() - t0)
    lines.append(dict(call="demcmc_power_posterior", rungs=K, rows=2000, particles=G * c["Np"], median_ms=1e3 * float(np.median(ts))))
    print(json.dumps(lines[0]), json.dumps(lines[-1]), sep="\n", flush=True)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        for ln in lines:
            f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Simulated (DEMCMC_SIMULATED) LBA likelihood on one GPU, next to the registered LBA kernel on the same data.

Workload: 2-accumulator LBA, N = 1000 trials, 4 groups x 256 particles, M in {2048, 8192, 16384} simulations per proposal,
and the registered LBA at the same N for context.  Per run: particle updates/s (CUDA events around the run call,
demcmc_counters.device_ms); from a second, separately timed pass (demcmc_set_timing time_loglik: CUDA events around every
likelihood launch) the k_ll_sim time per level, and two rates over that kernel time:
  nm_terms_per_s         N M per update, the size of the problem (an observation of label c meets only the m_c simulations
                         of its own label, so the kernel evaluates fewer terms than this);
  evaluated_terms_per_s  the Gaussian kernel terms k_ll_sim actually evaluates, sum_i m_(c_i) per update.  The timed pass is
                         repeated on a traced handle with the same seed (the same chain), and m_c is counted on the
                         simulations of SAMPLE proposals drawn from its trace, regenerated through demcmc_eval_simulated
                         under their run keys; evaluated_fraction = the mean of sum_i m_(c_i) / (N M) over them.
The fp64 share counts FP64_OPS_PER_TERM instructions per evaluated term (the SASS of k_ll_sim's inner loop as libnvrtc
12.9 compiles it: 16 DFMA, 4 DMUL, 3 DADD, 1 DSETP) against demcmc_fp64_peak (DFMA FLOP/s, two per instruction); the
simulations and the sort are not counted.  The first line names the card, its power limit and its maximum SM clock
(nvidia-smi, read only, in the same call).  One JSON line per run.

Usage: python scripts/bench_simulated.py [--out profiles/simulated_loglike_bench.jsonl] [--rounds 2]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import demcmc_b200 as D  # noqa: E402
from bench_configs import lba_sim_vec  # noqa: E402

INF = np.inf
FP64_OPS_PER_TERM = 24
SAMPLE = 256
LBA_SIM = """
#define DEMCMC_NPAR 5
__device__ void demcmc_prepare(const double *th, double *par) { for (int r = 0; r < 5; ++r) par[r] = th[r]; par[3] += th[2]; }
__device__ void demcmc_simulate(const double *par, demcmc_rng *rng, double *y)
{
    const double A = par[2], b = par[3];
    for (int tries = 0; tries < 1000; ++tries) {
        const double v1 = par[0] + demcmc_normal(rng), v2 = par[1] + demcmc_normal(rng);
        if (!(v1 > 0.0) && !(v2 > 0.0)) continue;
        const double t1 = v1 > 0.0 ? (b - A * demcmc_uniform(rng)) / v1 : DEMCMC_INF;
        const double t2 = v2 > 0.0 ? (b - A * demcmc_uniform(rng)) / v2 : DEMCMC_INF;
        y[0] = t1 <= t2 ? 1.0 : 2.0;
        y[1] = par[4] + (t1 <= t2 ? t1 : t2);
        return;
    }
    y[0] = 0.0; y[1] = DEMCMC_NAN;
}
"""


def _handle(impl, M, choice, rt, iters, trace=False):
    mn = float(rt.min())
    prior = [("normal", 1, 5), ("normal", 1, 5), ("normal", 0.8, 0.2), ("normal", 0.2, 0.1), ("uniform", 0, mn)]
    h = D.Handle(4, 256, 5, [0, 0, 0, 0, 0], [INF, INF, INF, INF, mn], seed=20261022, burnin=iters // 2, trace=trace)
    if impl == "registered":
        h.set_model("lba", prior, x=rt, choice=choice, n_dim=2)
    else:
        h.set_model("simulated", prior, x=np.column_stack([choice.astype(float), rt]), source=LBA_SIM, n_sim=M)
    r = np.random.default_rng(1)
    h.set_state(np.column_stack([np.abs(r.normal(2, 1, 1024)), np.abs(r.normal(2, 1, 1024)), np.abs(r.normal(0.8, 0.2, 1024)),
                                 np.abs(r.normal(0.2, 0.1, 1024)), r.uniform(0, mn, 1024)]))
    return h


def evaluated_fraction(M, choice, rt, warm, iters):
    """mean over SAMPLE proposals of the timed pass of sum_i m_(c_i) / (N M): the share of the N M terms k_ll_sim evaluates"""
    h = _handle("simulated", M, choice, rt, iters, trace=True)
    try:
        h.run(warm)
        h.run(iters)
        h.run(iters)                                                # the timed pass of run(): its proposals are in the trace
        tr = h.trace()
        S, P = tr["prop_weight"].shape
        pick = np.random.default_rng(3).choice(S * P, size=min(SAMPLE, S * P), replace=False)
        sweep = (warm + iters + pick // P).astype(np.uint32)        # one sweep per iteration (no blocks)
        unit = (pick % P).astype(np.uint32)                        # one device: global position = position
        _, sims = h.eval_simulated(tr["prop_theta"].reshape(-1, 5)[pick], sweep, unit, sims=True)
    finally:
        h.close()
    n_c = np.array([(choice == c).sum() for c in (1, 2)], dtype=float)
    val = sims[:, :, 1]
    m_c = np.stack([(np.isfinite(val) & (sims[:, :, 0] == c)).sum(axis=1) for c in (1, 2)], axis=1)
    return float(np.mean(m_c @ n_c) / (rt.size * M))


def run(impl, M, choice, rt, iters, peak):
    n = rt.size
    warm = max(2, iters // 10)
    h = _handle(impl, M, choice, rt, iters)
    try:
        h.run(warm)                                                 # warm-up: module load, allocations
        c0 = h.counters()
        h.run(iters)
        c1 = h.counters()
        h.set_timing(0, True)
        h.run(iters)
        c2 = h.counters()
    finally:
        h.close()
    ups = (c1["particle_updates"] - c0["particle_updates"]) / (c1["device_ms"] * 1e-3)
    out = {"workload": "lba", "impl": impl, "n_obs": n, "n_sim": M if impl == "simulated" else None, "particles": 1024, "iterations": iters,
           "particle_updates_per_s": ups, "ms_per_iteration": c1["device_ms"] / iters,
           "loglike_kernel_ms_per_iteration": c2["loglike_ms"] / iters,
           "loglike_kernel_ms_per_level": c2["loglike_ms"] / max(1, c2["levels"] - c1["levels"])}
    if impl == "simulated":
        upd = c2["particle_updates"] - c1["particle_updates"]
        nm = upd * n * M / (c2["loglike_ms"] * 1e-3)
        frac = evaluated_fraction(M, choice, rt, warm, iters)
        out.update({"nm_terms_per_s": nm, "end_to_end_nm_terms_per_s": ups * n * M, "evaluated_fraction": frac,
                    "evaluated_terms_per_s": nm * frac, "fp64_ops_per_term": FP64_OPS_PER_TERM, "fp64_peak_tflops": peak,
                    "share_of_fp64_peak": nm * frac * FP64_OPS_PER_TERM / (peak * 1e12 / 2)})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "simulated_loglike_bench.jsonl"))
    ap.add_argument("--rounds", type=int, default=2)
    a = ap.parse_args()
    D._ffi.use_library(D._ffi.DEFAULT_LIB)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    peak = D.fp64_peak(0)
    choice, rt = lba_sim_vec(np.random.default_rng(88484), 1000)
    lines = [{"nvidia_smi": smi.stdout.strip().splitlines(), "fp64_peak_tflops": peak}]
    print(json.dumps(lines[0]), flush=True)
    for _ in range(a.rounds):
        for impl, M, iters in (("registered", 0, 400), ("simulated", 2048, 40), ("simulated", 8192, 12), ("simulated", 16384, 6)):
            r = run(impl, M, choice, rt, iters, peak)
            lines.append(r)
            print(json.dumps(r), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for r in lines:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()

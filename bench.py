#!/usr/bin/env python
"""bench.py -- particle-updates/s of the DE-MCMC population step (BASELINE.json metric).

A "step" is one iteration of the sampler: migration (w.p. alpha) + one sweep over every particle
(proposal, full log-posterior, Metropolis accept, state/sample write).  Workload at N=1 is
BASELINE.json configs[1]: isotropic multivariate normal d=50, 1e5 observations, 4 groups x 256
particles, crossover + snooker (theta_snooker = 0.1), synthetic data (SURVEY.md 8d, seed 50514).
With N GPUs the groups shard over the ranks (4 groups per GPU, weak scaling) and migration crosses
NVLink through NCCL send/recv when a cycle spans ranks.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference ...                     # the CPU restatement of the reference
                                                           # (the reference is Julia; no Julia here)
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "particle-updates/sec (loglike evals incl.)"
UNIT = "particle-updates/s"
N_OBS, N_DIM, GROUPS_PER_GPU, NP = 100_000, 50, 4, 256
THETA_SNOOKER = 0.1
CONFIG_NAME = "BASELINE configs[1]"
L2_FLUSH_BYTES = 256 << 20


def workload_string():
    """config.workload: the same string on both arms (the driver compares them)"""
    return (f"isotropic MVN d={N_DIM}, {N_OBS} obs, {GROUPS_PER_GPU} groups x {NP} particles per GPU, "
            f"crossover+snooker {THETA_SNOOKER} ({CONFIG_NAME})")


def workload(n_groups, seed=50514):
    rng = np.random.default_rng(seed)
    mu = rng.normal(size=N_DIM)
    x = rng.normal(mu, 1.0, size=(N_OBS, N_DIM))
    prior = [("normal", 0.0, 1.0)] * N_DIM + [("halfcauchy", 0.0, 1.0)]
    lo = [-np.inf] * N_DIM + [0.0]
    hi = [np.inf] * (N_DIM + 1)
    # initial states: prior draws as in the example's sample_prior (Multivariate_Guassian_Example.jl:16-20)
    P = n_groups * NP
    theta0 = np.column_stack([rng.normal(size=(P, N_DIM)), np.abs(rng.standard_cauchy(P))])
    return x, prior, lo, hi, theta0


class ClockSampler:
    """SM clock and clock-event (throttle) reasons sampled DURING the timed region (B200_PROFILING.md):
    NVML polled every 2 ms from a thread of this process (the timed region of a short run is a few
    tens of milliseconds -- `nvidia-smi -lms 100` would not land one sample in it); nvidia-smi is the
    fallback when NVML cannot be loaded."""
    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"),
               (0x80, "hw_power_brake_slowdown"))

    def __init__(self, index, uuid=None):
        self.index, self.uuid, self.rows, self.stop_flag, self.thread, self.src = index, uuid, [], False, None, None
        self.nv = self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            if uuid:
                for u in (f"GPU-{uuid}", str(uuid)):
                    try:
                        h = pynvml.nvmlDeviceGetHandleByUUID(u)
                        break
                    except Exception:
                        h = None
            if h is None:
                vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
                ids = [v for v in vis.split(",") if v.strip().isdigit()]
                h = pynvml.nvmlDeviceGetHandleByIndex(int(ids[index]) if index < len(ids) else index)
            self.nv, self.h, self.src = pynvml, h, "nvml"
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = self.h = None

    def _poll_nvml(self):
        nv, h = self.nv, self.h
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop_flag:
            try:
                self.rows.append((time.time(), float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), int(get_reasons(h))))
            except Exception:
                pass
            time.sleep(0.002)

    def _poll_smi(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.active"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.max_mhz = float(out[1])
                self.rows.append((time.time(), float(out[0]), int(out[2].strip(), 16)))
            except Exception:
                time.sleep(0.05)

    def start(self):
        if self.nv is None:
            self.src, self.max_mhz = "nvidia-smi", None
        self.thread = threading.Thread(target=self._poll_nvml if self.nv is not None else self._poll_smi, daemon=True)
        self.thread.start()

    def stop(self, windows):
        """windows: [(t0, t1, label)] of GPU-busy passes of the same workload; the first is the timed region."""
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=6)
        t0, t1, _ = windows[0]
        timed = [r for r in self.rows if t0 <= r[0] <= t1]
        used, where = timed, "timed region"
        if not used:                                  # region shorter than one poll: the identical passes that follow it
            used = [r for r in self.rows if any(a <= r[0] <= b for a, b, _ in windows)]
            where = "timed region + the identical passes after it"
        sm = [r[1] for r in used]
        bits = 0
        for r in used:
            bits |= r[2]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_min_mhz": min(sm) if sm else None,
                "sm_max_mhz": self.max_mhz, "reasons": [n for b, n in self.REASONS if bits & b],
                "samples": len(sm), "samples_in_timed_region": len(timed), "window": where, "source": self.src}


def ncu_traffic(persistent=False):
    """dram bytes read + written per launch of the dominant kernel from the committed `ncu --set full` capture."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r02_k_chunk_persist_traffic.json" if persistent else "r01_k_xdot_traffic.json")))
        return t["dram_bytes_read_per_launch"] + t["dram_bytes_write_per_launch"]
    except (OSError, KeyError, ValueError):
        return None


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        return {}


DUMP_LIMIT_BYTES = 60 << 20       # --dump-outputs: below 64 MB in all, .npy headers included


def last_chain_row(h, world=1, rank=0):
    """The last stored row of the chains as sample() returns it, [P][d + 2] with one row per particle id of the whole job.
    A sharded handle has no chains of its own: every rank sends its last row by position to rank 0, which merges the
    rows by particle id as distributed.sample() does (None on the other ranks)."""
    if world == 1:
        return h.chains(h.stored_iterations - 1, 1)[:, :, 0]
    import torch.distributed as dist

    from demcmc_b200 import distributed
    parts = distributed._gather_arrays(dist, h.history_by_slot(h.stored_iterations - 1, 1), rank, world, h.cfg.device)
    if rank != 0:
        return None
    th, w, ids, acc = (p if isinstance(p, np.ndarray) else p.cpu().numpy() for p in parts)
    samples, lp, accept, final_ids = distributed._merge_by_id(th, w, ids, acc, 1, h.P_total, h.d)
    return np.column_stack([samples[:, :, 0], accept[final_ids, 0], lp[final_ids, 0]])


def dump_outputs(out_dir, row):
    """Writes what the timed run left for a caller, so that two builds can be compared output for output: `row`, the
    last_chain_row() of the run, split into the parameters, the acceptance flags and the log posteriors, float64.  When
    it exceeds DUMP_LIMIT_BYTES, a fixed, seeded sample of the particle ids is written; particle_id.npy names the ids
    either way."""
    ids = np.arange(row.shape[0])
    if row.nbytes + ids.size * 8 > DUMP_LIMIT_BYTES:
        ids = np.sort(np.random.default_rng(0).choice(ids.size, DUMP_LIMIT_BYTES // ((row.shape[1] + 1) * 8), replace=False))
        row = row[ids]
    os.makedirs(out_dir, exist_ok=True)
    d = row.shape[1] - 2
    for name, a in (("samples", row[:, :d]), ("acceptance", row[:, d]), ("lp", row[:, d + 1]), ("particle_id", ids)):
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a, dtype=np.float64))


# ---------------------------------------------------------------------------------------------
# CPU arm: the C restatement of the reference's algorithm (oracle/), one thread per group as the
# reference's ThreadsX.map over groups (src/main.jl:135-148)
# ---------------------------------------------------------------------------------------------
def cpu_updates_per_s(steps, warmup, budget_s=100.0):
    from oracle import oracle as O
    O.set_plain_sums(True)     # the timing variant of the restatement: plain fp64 sums, not the compensated ones of the parity oracle
    x, prior, lo, hi, _ = workload(GROUPS_PER_GPU)
    model = O.Model("mvnormal", N_DIM + 1, prior, x=x)
    cores = min(GROUPS_PER_GPU, os.cpu_count() or 1)
    rng = np.random.default_rng(1)

    def run(np_sample, n_iter):
        P = GROUPS_PER_GPU * np_sample
        theta0 = np.column_stack([rng.normal(size=(P, N_DIM)), np.abs(rng.standard_cauchy(P)) + 0.5])
        cfg = O.Config(GROUPS_PER_GPU, np_sample, N_DIM + 1, lo, hi, burnin=0, theta_snooker=THETA_SNOOKER, n_threads=cores, seed=3)
        t0 = time.perf_counter()
        O.run(cfg, model, theta0, n_iter, record=False, trace=False, history=False)
        return time.perf_counter() - t0, P * n_iter

    # probe the per-update cost, then size the per-step sample so the whole run fits the budget
    t, n = run(3, 1)
    per_update = (t - 0.0) / (n + GROUPS_PER_GPU * 3)      # the run also evaluates the initial weights
    total = max(1, steps + warmup)
    np_sample = int(max(3, min(NP, budget_s / (per_update * total * GROUPS_PER_GPU))))
    if warmup > 0:
        run(np_sample, min(warmup, 1))
    t, n = run(np_sample, steps)
    t_init = per_update * GROUPS_PER_GPU * np_sample        # initial-weight evaluations are not updates
    ups = n / max(t - t_init, 1e-9)
    sample = (f"{steps} iterations of the same model/data (d={N_DIM}, {N_OBS} obs, {GROUPS_PER_GPU} groups) with "
              f"{np_sample} particles per group" + ("" if np_sample == NP else f" instead of {NP}") + f" ({n} particle updates)")
    return ups, cores, sample, t / max(1, steps) * 1e3


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ups, cores, sample, ms = cpu_updates_per_s(args.steps, args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": ups, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_string(), "groups_total": GROUPS_PER_GPU, "particles_total": GROUPS_PER_GPU * NP,
                       "note": "the CPU arm always runs ONE GPU's share of the job (4 groups): at --gpus N > 1 the B200 arm runs N times as many groups, so only the N = 1 ratio compares like with like"},
            "cpu_baseline": {"value": ups, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                             "note": "C restatement of the reference's algorithm (oracle/) with plain fp64 sums, one thread per group = the reference's own parallel width (ThreadsX.map over groups, src/main.jl:135-148); the reference itself is Julia and cannot run in this image (julia/cpu_baseline.jl is the script for where it can)"},
            "e2e": {"value": ups, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist

    import demcmc_b200 as D

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; libdemcmc_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    # stdout carries the one JSON line only: whatever a library prints there (NCCL's version banner,
    # for one) goes to stderr -- file descriptor 1 points at stderr until the line is printed
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    D._ffi.use_library(D._ffi.DEFAULT_LIB)
    assert D._ffi.lib().demcmc_backend_name() == b"cuda-sm100a"

    G = GROUPS_PER_GPU * world
    x, prior, lo, hi, theta0 = workload(G)
    P_local = GROUPS_PER_GPU * NP
    d = N_DIM + 1
    kw = dict(burnin=0, theta_snooker=THETA_SNOOKER, seed=20261017, device=local, group_begin=rank * GROUPS_PER_GPU,
              group_count=GROUPS_PER_GPU)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- kernel-side number: inputs resident in HBM before the timed region ----------------------
    xd = torch.from_numpy(x).to(f"cuda:{local}")                      # the data set, already on the device
    torch.cuda.synchronize()
    h = D.Handle(G, NP, d, lo, hi, **kw)
    h.set_model("mvnormal", prior, device_ptrs=(xd.data_ptr(), None), n_obs=N_OBS, n_dim=N_DIM)
    if world > 1:
        uid = [D.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        h.comm_init(uid[0], rank, world)
    h.set_state(theta0[rank * P_local:(rank + 1) * P_local])
    h.set_timing(L2_FLUSH_BYTES, False)
    h.run(args.warmup)
    c0 = h.counters()
    try:
        uuid = str(torch.cuda.get_device_properties(local).uuid)
    except Exception:
        uuid = None
    # rank 0 samples its GPU (the line reports rank 0's clocks); NVML queries take a driver-wide lock, and eight
    # processes polling at 500 Hz each get in the way of each other's kernel launches
    clocks = ClockSampler(local, uuid) if rank == 0 else None
    if clocks:
        clocks.start()
    barrier()
    t0 = time.time()
    h.run(args.steps)
    barrier()
    t1 = time.time()
    c1 = h.counters()
    if args.dump_outputs:
        row = last_chain_row(h, world, rank)                         # every rank takes part in the gather
        if rank == 0:
            dump_outputs(args.dump_outputs, row)
    windows = [(t0, t1, "timed")]
    wall_timed = t1 - t0
    # second pass of the same length with every likelihood launch bracketed by CUDA events on the
    # launching stream (this is what the roofline of the dominant kernel is computed from; the
    # events between kernels switch off the programmatic-dependent-launch overlap of the first pass)
    h.set_timing(L2_FLUSH_BYTES, True)
    barrier()
    tw = time.time()
    h.run(args.steps)
    barrier()
    windows.append((tw, time.time(), "roofline pass"))
    c2 = h.counters()
    ms = torch.tensor([c1["device_ms"]], dtype=torch.float64, device=f"cuda:{local}")
    ms_ll = torch.tensor([c2["loglike_ms"]], dtype=torch.float64, device=f"cuda:{local}")
    ms_pass2 = torch.tensor([c2["device_ms"]], dtype=torch.float64, device=f"cuda:{local}")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)                    # max over ranks, device time
        dist.all_reduce(ms_ll, op=dist.ReduceOp.MAX)
        dist.all_reduce(ms_pass2, op=dist.ReduceOp.MAX)
    ms, ms_ll, ms_pass2 = float(ms.item()), float(ms_ll.item()), float(ms_pass2.item())
    updates = (c1["particle_updates"] - c0["particle_updates"]) * world
    launches = c1["kernel_launches"] - c0["kernel_launches"]
    persistent = (c2["persistent_chunks"] - c1["persistent_chunks"]) > 0
    ll_launches = (c2["persistent_chunks"] - c1["persistent_chunks"]) if persistent else (c2["levels"] - c1["levels"])
    ll_levels = c2["levels"] - c1["levels"]
    value = updates / (ms * 1e-3)

    # steady state without the L2 flush (how a real run behaves: the data set stays in L2)
    h.set_timing(0, False)
    barrier()
    tw = time.time()
    h.run(args.steps)
    barrier()
    windows.append((tw, time.time(), "steady pass"))
    ms_steady = torch.tensor([h.counters()["device_ms"]], dtype=torch.float64, device=f"cuda:{local}")
    if world > 1:
        dist.all_reduce(ms_steady, op=dist.ReduceOp.MAX)
    ms_steady = float(ms_steady.item())
    c3 = h.counters()
    # SURVEY hard part 7, reported separately: with the data centred on their column means the streamed cross term is
    # analytically zero, so the same chain follows from O(d) sufficient statistics -- the O(N d) stream skipped
    ms_suff = None
    if world == 1:
        h.set_sufficient_stat(True)
        h.run(args.warmup)
        barrier()
        tw = time.time()
        h.run(args.steps)
        barrier()
        windows.append((tw, time.time(), "sufficient-statistic pass"))
        ms_suff = h.counters()["device_ms"]
        h.set_sufficient_stat(False)
    ck = clocks.stop(windows) if clocks else None
    h.close()

    # ---- roofline of the dominant kernel (k_ssd, the likelihood) ----------------------------------
    peaks = measured_peaks()
    dfma_peak, dmma_peak = D.fp64_peaks(local)                       # fp64 microbenchmarks, TFLOP/s (not in MEASURED_PEAKS.json)
    fp64_peak = max(dfma_peak, dmma_peak)
    flops = 2.0 * N_OBS * N_DIM * (updates / world)                  # contraction form: one DFMA per (obs, dim, particle)
    achieved = flops / (ms_ll * 1e-3) / 1e12 if ms_ll > 0 else None
    kname = ("k_chunk_persist (persistent, warp-specialised: DMMA likelihood + proposals + accepts of all levels of a chunk of <= 16 steps)"
             if persistent else "k_xdot<MVN>")
    measured_in = (("a second pass of the same steps with CUDA events around every k_chunk_persist launch (one launch per chunk; "
                    "%d dependency levels in %d launches; ms_per_step of that pass: %.4f)" % (ll_levels, ll_launches, ms_pass2 / args.steps))
                   if persistent else
                   "a second pass of the same steps with CUDA events around every k_xdot launch (ms_per_step of that pass: %.4f)" % (ms_pass2 / args.steps))
    roofline = {"bound": "tensor", "pipe": "fp64 tensor path (DMMA m8n8k4)", "kernel": kname, "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s",
                "frac": achieved / fp64_peak if achieved else None,
                "traffic": ncu_traffic(persistent),
                "algorithmic_flops_per_launch": flops / max(1, ll_launches), "launches": ll_launches,
                "avg_launch_ms": ms_ll / max(1, ll_launches), "share_of_step": ms_ll / ms_pass2 if ms_pass2 > 0 else None,
                "measured_in": measured_in,
                "peak_source": "measured in this run (MEASURED_PEAKS.json has no fp64 entry): the larger of a DFMA loop and a DMMA m8n8k4 loop, 8 warps x 8 CTAs/SM; the two fp64 paths share one pipe on B200",
                "peak_dfma": dfma_peak, "peak_dmma": dmma_peak,
                "note": "bound = the fp64 tensor path (DMMA m8n8k4; peak = this run's fp64 microbenchmarks, not the bf16 figure of MEASURED_PEAKS.json): ~400 flop/B against the L2-resident data set; algorithmic work = 2*N*d flop per particle update (one multiply-add per observation x dimension x particle, contraction form of the sum of squares); padding of d to whole k-steps of 4 and of levels to whole octets of particles is NOT counted as work; for the persistent kernel the duration includes the proposals and accepts it runs (the scalar SMs do only those). WHAT THE STREAM COMPUTES: the kernel centres the data on their exact column means, so the streamed cross term B = sum_i sum_k x'_ik m'_k is analytically ZERO and the log-likelihood rests on the O(d) terms sum x'^2 and n sum m'^2; every observation is streamed for every particle only because the metric counts 'loglike evals incl.' (SURVEY hard part 7) -- value_sufficient_stat is the same chain with the stream skipped. The kernel's arithmetic is pinned on operands whose answer is not zero by tests/test_gpu_xdot.py (caller-supplied centre, B against an extended-precision reference to 2^-40 of its Cauchy-Schwarz bound, both launch paths, mutation tests)",
                "hbm_gbs_measured": peaks.get("hbm_gbs")}

    # ---- end to end through the public API with HOST buffers -------------------------------------
    e2e = None
    if rank == 0 or world > 1:
        rng = np.random.default_rng(7)
        # the caller's observations sit in page-locked host memory (the contract's "host->device copy ... from pinned host
        # memory"): the library's upload is then one DMA instead of the driver's staged pageable path
        x_host = torch.from_numpy(x).pin_memory().numpy()
        model = D.DEModel(sample_prior=lambda: [rng.normal(size=N_DIM), abs(rng.standard_cauchy())],
                          prior_loglike=D.GPUPrior(D.Normal(0, 1), D.HalfCauchy(0, 1)),
                          loglike=D.GPULoglike("mvnormal", x_host), names=("μ", "σ"))
        if world == 1:
            de = D.DE(sample_prior=model.sample_prior, bounds=((-np.inf, np.inf), (0.0, np.inf)), n_groups=G, Np=NP, burnin=0,
                      θsnooker=THETA_SNOOKER, seed=11)
            # one untimed call of the same size first: it warms the context, the device pool and -- what
            # matters most on a fresh VM -- the host pages the chains land in (first touch of never-used
            # guest memory made the download of the same 217 MB take anything from 0.04 s to 2.2 s)
            D.sample(model, de, args.steps, device=local)
            torch.cuda.synchronize()
            # where the call spends its time (reported next to the number, not used by it)
            parts = {}

            def timed(cls, name):
                orig = getattr(cls, name)

                def wrapper(*a, **k):
                    t = time.perf_counter()
                    try:
                        return orig(*a, **k)
                    finally:
                        parts[name] = parts.get(name, 0.0) + time.perf_counter() - t
                setattr(cls, name, wrapper)
                return orig
            saved = {n: timed(D.Handle, n) for n in ("set_model", "set_state", "run", "chains")}
            t0 = time.perf_counter()
            chains = D.sample(model, de, args.steps, device=local)   # host data in, chains out
            t_e2e = time.perf_counter() - t0
            for n, f in saved.items():
                setattr(D.Handle, n, f)
            assert len(chains) == args.steps
            h2d = (x.nbytes + G * NP * d * 8) / args.steps
            d2h = G * NP * (d + 2) * 8
            e2e = {"value": G * NP * args.steps / t_e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                   "call": "sample(model, de, n_iter) with the observations in pinned host memory (numpy view): handle creation, data upload + packing, P sample_prior() calls, all iterations, device-side bundle_samples and the download of the chains into a fresh numpy array; timed on the second call of the process",
                   "seconds": t_e2e, "seconds_by_part": {k: round(v, 4) for k, v in parts.items()}}
    if world > 1:
        # sharded e2e through the user-facing call: every rank calls distributed.sample(model, de, n_iter) with HOST data;
        # rank 0 gets the Chains (per-rank by-slot histories gathered and merged by id on the host)
        from demcmc_b200 import distributed

        def make():
            r = np.random.default_rng(7)
            m = D.DEModel(sample_prior=lambda: [r.normal(size=N_DIM), abs(r.standard_cauchy())],
                          prior_loglike=D.GPUPrior(D.Normal(0, 1), D.HalfCauchy(0, 1)), loglike=D.GPULoglike("mvnormal", x_host), names=("μ", "σ"))
            return m, D.DE(sample_prior=m.sample_prior, bounds=((-np.inf, np.inf), (0.0, np.inf)), n_groups=G, Np=NP, burnin=0, θsnooker=THETA_SNOOKER, seed=11)
        m_, de_ = make()
        distributed.sample(m_, de_, args.steps, device=local)      # untimed, SAME size: contexts, pools, NCCL buffers and host pages of the timed call (a shorter warm-up left one 4-GPU run at 104 ms instead of 34)
        m_, de_ = make()
        barrier()
        t0 = time.perf_counter()
        chains = distributed.sample(m_, de_, args.steps, device=local)
        barrier()
        t_e2e = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=f"cuda:{local}")
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
        t_e2e = float(t_e2e.item())
        if rank == 0:
            assert len(chains) == args.steps and chains.value.shape[2] == G * NP
        e2e = {"value": G * NP * args.steps / t_e2e, "unit": UNIT, "h2d_bytes_per_step": (x.nbytes + P_local * d * 8) / args.steps,
               "d2h_bytes_per_step": P_local * (d * 8 + 8 + 4 + 1), "seconds": t_e2e,
               "call": "distributed.sample(model, de, n_iter) on every rank with host (numpy) data: handle creation, data upload + packing, the P sample_prior() draws "
                       "on rank 0 and their broadcast, all iterations (migration across ranks included), the download of every rank's history, the gather on rank 0 and the "
                       "by-id merge into the Chains; max over ranks of the wall time between two barriers, second call of the process",
               "migration": distributed.last_counters and {k: distributed.last_counters[k] for k in ("cross_migrations", "mailbox_events")}}

    # ---- ESS/s, the second half of BASELINE.json's metric: a fixed-length leg, whatever --steps is -----------------------
    if rank == 0 and world == 1 and not args.no_ess:
        from demcmc_b200.diagnostics import bulk_ess
        n_ess, burn_ess = 1000, 400
        xbar = x.mean(axis=0)
        s_pool = float(np.sqrt(((x - xbar) ** 2).sum() / x.size))
        r3 = np.random.default_rng(13)
        # chains started around the posterior mode (xbar +- a posterior sd): from N(0,1) prior draws this model needs
        # thousands of iterations before any draw is usable (d = 51, posterior sd 0.003); the ESS of unconverged chains says nothing
        m3 = D.DEModel(sample_prior=lambda: [xbar + r3.normal(0, s_pool / np.sqrt(N_OBS), N_DIM), s_pool * (1 + r3.normal(0, 5e-4))],
                       prior_loglike=D.GPUPrior(D.Normal(0, 1), D.HalfCauchy(0, 1)), loglike=D.GPULoglike("mvnormal", x_host), names=("μ", "σ"))
        de3 = D.DE(sample_prior=m3.sample_prior, bounds=((-np.inf, np.inf), (0.0, np.inf)), n_groups=G, Np=NP, burnin=burn_ess, θsnooker=THETA_SNOOKER, seed=17)
        # (like the e2e leg: one untimed call of the same size first -- the first touch of the 260 MB of host pages the chains land
        # in is the guest VM's cost, 0.3 s on a fresh box, and made this leg read 1.5 k or 2.6 k ESS/s depending on what ran before it)
        D.sample(m3, de3, n_ess, device=local)
        r3 = np.random.default_rng(13)
        t0 = time.perf_counter()
        ch3 = D.sample(m3, de3, n_ess, device=local)
        t_ess = time.perf_counter() - t0
        ess = np.array([bulk_ess(ch3.value[:, k, :]) for k in range(d)])
        from demcmc_b200.diagnostics import split_rhat
        rhat = np.array([split_rhat(ch3.value[:, k, :]) for k in range(0, d, 10)])
        if e2e is None:
            e2e = {}
        e2e["ess"] = {"min_bulk_ess": float(np.nanmin(ess)), "median_bulk_ess": float(np.nanmedian(ess)), "ess_per_s": float(np.nanmin(ess)) / t_ess,
                      "seconds": t_ess, "iterations": n_ess, "burnin_discarded": burn_ess, "draws": int(ch3.value.shape[0]), "chains": int(ch3.value.shape[2]),
                      "max_split_rhat_sampled": float(np.nanmax(rhat)),
                      "note": "ESS/s = min over the 51 parameters of the rank-normalised split bulk ESS (Vehtari et al. 2021) of the kept draws, all chains pooled, "
                              "divided by the wall time of the WHOLE sample() call (host data in, burn-in iterations included, chains out); 1000 iterations of which the "
                              "first 400 are discarded; chains started around the posterior mode (a cold start from the N(0,1) prior needs thousands of iterations "
                              "at d = 51 with posterior sd 0.003)"}

    # ---- the other BASELINE shapes, one GPU (scripts/bench_configs.py): driver-observed companion numbers -----------------
    configs = None
    if rank == 0 and world == 1 and not args.no_configs:
        sys.path.insert(0, os.path.join(ROOT, "scripts"))
        import bench_configs
        configs = []
        for name in ("c1", "c3", "c4", "c5"):
            try:
                configs.append(bench_configs.run(name, peaks=(dfma_peak, dmma_peak), hbm_gbs=peaks.get("hbm_gbs")))
            except Exception as e:                                   # a companion number must never cost the headline line
                configs.append({"config": name, "error": repr(e)})

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        ups, cores, sample, _ = cpu_updates_per_s(2, 0, budget_s=25.0)
        cpu = {"value": ups, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic",
                "config": {"workload": workload_string(),
                           "groups_total": G, "particles_total": G * NP, "parallelism": f"groups sharded over {world} GPU(s); NCCL send/recv migration",
                           "l2": f"flushed: {L2_FLUSH_BYTES >> 20} MiB overwritten before every segment = a migration (with its NCCL exchange) plus the chunk of overlapped steps that follows it (a chunk ends at the next migration, at most 16 steps; steps inside a chunk share launches so there is no per-step boundary); per-segment CUDA events, flush excluded",
                           "timing": "CUDA events on the library's launching stream (demcmc_counters.device_ms), max over ranks"},
                "value_steady_no_flush": updates / (ms_steady * 1e-3),
                "value_sufficient_stat": (c3["particle_updates"] - c2["particle_updates"]) / (ms_suff * 1e-3) if ms_suff else None,
                "value_sufficient_stat_note": "the same chain with the O(N d) stream skipped (demcmc_set_sufficient_stat; exact: the cross term is analytically zero with mean-centred data); NOT the headline: the metric counts log-likelihood evaluations that stream every observation" if ms_suff else None,
                "configs": configs,
                "gpu_launches": int(launches), "clocks": ck, "roofline": roofline, "e2e": e2e, "cpu_baseline": cpu,
                "wall_s_timed_region": wall_timed}
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if world > 1:
        dist.destroy_process_group()


def run_single_process(args):
    """The same workload, N GPUs, ONE process: what a Julia caller of sample(model, de, n_iter; devices = 0:N-1) gets."""
    import torch

    import demcmc_b200 as D
    D._ffi.use_library(D._ffi.DEFAULT_LIB)
    N = args.gpus
    G = GROUPS_PER_GPU * N
    x, prior, lo, hi, theta0 = workload(G)
    d = N_DIM + 1
    h = D.Handle(G, NP, d, lo, hi, burnin=0, theta_snooker=THETA_SNOOKER, seed=20261017, devices=list(range(N)))
    h.set_model("mvnormal", prior, x=x)
    h.set_state(theta0)
    h.set_timing(L2_FLUSH_BYTES, False)
    h.run(args.warmup)
    c0 = h.counters()
    t0 = time.perf_counter()
    h.run(args.steps)
    wall = time.perf_counter() - t0
    c1 = h.counters()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_chain_row(h))
    h.set_timing(0, False)
    h.run(args.steps)
    c2 = h.counters()
    h.close()
    updates = c1["particle_updates"] - c0["particle_updates"]
    rng = np.random.default_rng(7)
    model = D.DEModel(sample_prior=lambda: [rng.normal(size=N_DIM), abs(rng.standard_cauchy())], prior_loglike=D.GPUPrior(D.Normal(0, 1), D.HalfCauchy(0, 1)),
                      loglike=D.GPULoglike("mvnormal", x), names=("μ", "σ"))
    de = D.DE(sample_prior=model.sample_prior, bounds=((-np.inf, np.inf), (0.0, np.inf)), n_groups=G, Np=NP, burnin=0, θsnooker=THETA_SNOOKER, seed=11)
    D.sample(model, de, args.steps, devices=list(range(N)))             # untimed, same size as the timed call
    t0 = time.perf_counter()
    chains = D.sample(model, de, args.steps, devices=list(range(N)))
    t_e2e = time.perf_counter() - t0
    assert chains.value.shape == (args.steps, d + 2, G * NP)
    line = {"metric": METRIC, "value": updates / (c1["device_ms"] * 1e-3), "unit": UNIT, "n_gpus": N, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": c1["device_ms"] / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_string(), "groups_total": G, "particles_total": G * NP,
                       "parallelism": f"ONE process, one multi-device handle over {N} GPU(s): a host thread per GPU, migration through peer-mapped mailboxes",
                       "timing": "device_ms = the slowest device's CUDA-event time (L2 flushed between segments)"},
            "value_wall": updates / wall, "value_steady_no_flush": (c2["particle_updates"] - c1["particle_updates"]) / (c2["device_ms"] * 1e-3),
            "gpu_launches": int(c1["kernel_launches"] - c0["kernel_launches"]),
            "migration": {"cross_device": int(c1["cross_migrations"] - c0["cross_migrations"]), "through_mailboxes": int(c1["mailbox_events"] - c0["mailbox_events"])},
            "e2e": {"value": G * NP * args.steps / t_e2e, "unit": UNIT, "seconds": t_e2e, "h2d_bytes_per_step": (N * x.nbytes + G * NP * d * 8) / args.steps,
                    "d2h_bytes_per_step": G * NP * (d + 2) * 8, "call": "sample(model, de, n_iter, devices=[0..N-1]) from one process, host data in, Chains out"}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--no-ess", action="store_true", help="skip the ESS/s leg")
    ap.add_argument("--no-configs", action="store_true", help="skip the companion numbers of the other BASELINE shapes")
    ap.add_argument("--single-process", action="store_true",
                    help="python bench.py --gpus N --single-process: ONE process drives the N GPUs through a multi-device handle (demcmc_config.n_devices) instead of one torchrun rank per GPU")
    # the same step on another BASELINE shape (the contract's line is the default, configs[1]); configs[4] is
    # --dim 100 --particles 4096 --groups-per-gpu 8 on 8 GPUs
    ap.add_argument("--dim", type=int, default=None, help="dimensions of the multivariate normal (default 50)")
    ap.add_argument("--particles", type=int, default=None, help="particles per group (default 256)")
    ap.add_argument("--groups-per-gpu", type=int, default=None, help="groups per GPU (default 4)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the chains' last row (parameters, acceptance, lp) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the B200 arm computed; the reference arm runs fewer particles")
    global N_DIM, NP, GROUPS_PER_GPU
    shape_given = args.dim or args.particles or args.groups_per_gpu
    N_DIM, NP, GROUPS_PER_GPU = args.dim or N_DIM, args.particles or NP, args.groups_per_gpu or GROUPS_PER_GPU
    if shape_given:
        global CONFIG_NAME
        CONFIG_NAME = ("BASELINE configs[4]: 64 groups x 4096 across 8 GPUs" if (N_DIM, NP, GROUPS_PER_GPU, args.gpus) == (100, 4096, 8, 8)
                       else "a shape given on the command line, not a BASELINE config")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    elif args.single_process:
        run_single_process(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()

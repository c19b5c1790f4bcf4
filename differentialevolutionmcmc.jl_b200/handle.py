"""Thin object wrapper over the C ABI handle (one per process / GPU)."""
from __future__ import annotations

import ctypes as C

import os

import numpy as np

from . import _ffi
from ._ffi import _bp, _dp, _ip, check, f8, ptr

KINDS = {"gaussian": 0, "mvnormal": 1, "binomial": 2, "lnr": 3, "lba": 4, "hier_normal": 5, "rastrigin": 6, "mvnormal_full": 7,
         "custom": 8, "simulated": 9}
UPDATES = {"mh": 0, "maximize": 1, "minimize": 2}
FITNESS = {"posterior": 0, "fun": 1}
PRIORS = {"flat": 0, "normal": 1, "halfcauchy": 2, "uniform": 3, "beta": 4, "normal_ref": 5}
PROPOSALS = {"random_gamma": 0, "fixed_gamma": 1, "variable_gamma": 2}


def _out_empty(shape):
    """The array a large download lands in.  DEMCMC_PINNED_OUT=1: page-locked memory from torch's caching host allocator, which
    the copy engine writes directly -- worth it only for callers that drop each result before the next call (the allocator
    can then reuse the block; pinning a fresh 222 MB block costs 115 ms, five times the pageable download).  Default: numpy
    memory through the library's pipelined staging copy."""
    n = int(np.prod(shape))
    if n * 8 >= (1 << 20) and os.environ.get("DEMCMC_PINNED_OUT", "0") == "1":
        try:
            import torch
            if torch.cuda.is_available():
                return torch.empty(n, dtype=torch.float64, pin_memory=True).numpy().reshape(shape)
        except Exception:                                    # noqa: BLE001 -- no torch, no CUDA runtime in torch: pageable
            pass
    return np.empty(shape)


class Handle:
    """demcmc_handle: the DE sampler bound to one GPU (or to a shard of the groups)."""

    def __init__(self, n_groups, Np, d, lo, hi, burnin=1000, n_initial=0, alpha=0.1, beta=0.1, eps=0.001,
                 sigma=0.05, kappa=1.0, theta_snooker=0.0, proposal="random_gamma", blocks=None, seed=0,
                 device=0, group_begin=0, group_count=0, trace=False, store_every=1, resample=False, update="mh", fitness="posterior",
                 blocking_schedule=None, devices=None):
        """devices=[0, 1, ...]: ONE handle over several GPUs of the box from this one process (cfg.n_devices)."""
        self._h = C.c_void_p()
        self.devices = None if devices is None or len(devices) <= 1 else np.ascontiguousarray(devices, dtype=np.int32)
        if devices is not None and len(devices) == 1:
            device = int(devices[0])
        self.lo, self.hi = f8(lo), f8(hi)
        if self.lo.shape != (d,) or self.hi.shape != (d,):
            raise ValueError("bounds must be expanded to one (lo, hi) per flattened parameter")
        self.blocks = None if blocks is None else np.ascontiguousarray(blocks, dtype=np.uint8).reshape(-1, d)
        nb = 0 if self.blocks is None else self.blocks.shape[0]
        prop = PROPOSALS[proposal] if isinstance(proposal, str) else int(proposal)
        self.cfg = _ffi.Config(_ffi.ABI_VERSION, n_groups, Np, d, burnin, n_initial, alpha, beta, eps, sigma, kappa,
                               theta_snooker, prop, nb, ptr(self.blocks, _bp), ptr(self.lo, _dp), ptr(self.hi, _dp),
                               int(seed) & (2**64 - 1), device, group_begin, group_count, int(bool(resample)), int(bool(trace)), store_every,
                               UPDATES[update], FITNESS[fitness], 0 if self.devices is None else self.devices.size, ptr(self.devices, _ip))
        self.n_groups, self.Np, self.d = n_groups, Np, d
        self.G_local = group_count if group_count > 0 else n_groups
        self.P = self.G_local * Np
        self.P_total = n_groups * Np
        self.B = max(1, nb)
        self.n_initial = n_initial
        self.n_obs = 0                                      # observations of the bound model (set_model)
        self.store_every = max(1, int(store_every))
        self.iterations = 0
        self._last_iters = 0
        self._keep = []
        check(_ffi.lib().demcmc_create(C.byref(self.cfg), C.byref(self._h)))
        if blocking_schedule is not None:
            self.set_blocking_schedule(blocking_schedule)

    def close(self):
        if self._h:
            _ffi.lib().demcmc_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- model ---------------------------------------------------------------------------------
    def set_model(self, kind, prior, x=None, choice=None, sigma=None, lba_floor=1e-10, device_ptrs=None, n_obs=None,
                  n_dim=0, n_per=0, center=None, cov=None, source=None, n_cols=None, n_sim=0, sim_floor=1e-10):
        """Bind a registered likelihood kernel.  `prior` is a list of (name, a, b, ref) per
        flattened parameter.  `device_ptrs=(x_ptr, choice_ptr)` passes data already in HBM.
        kind="custom": `source` is the CUDA C++ text of the likelihood (include/demcmc_b200.h: DEMCMC_CUSTOM) and x an
        n_obs-vector (n_cols = 1), an n_obs x n_cols matrix, or None (no observations); with device pointers pass
        n_obs and n_cols.
        kind="simulated": `source` is the CUDA C++ text of the simulator (include/demcmc_b200.h: DEMCMC_SIMULATED), x an
        n_obs-vector of values (n_cols = 1) or an n_obs x 2 matrix of (label, value) rows, n_sim the simulations per proposal
        and sim_floor the density floor.
        `center` (mvnormal / hier_normal, test hook): centre the data on this vector instead of on their
        column means, which makes the streamed cross term non-zero (demcmc_model.center)."""
        d = self.d
        if len(prior) != d:
            raise ValueError(f"need {d} prior specs, got {len(prior)}")
        pr = (_ffi.Prior * d)()
        for k, p in enumerate(prior):
            pr[k] = _ffi.Prior(PRIORS[p[0]], int(p[3]) if len(p) > 3 else 0, float(p[1]) if len(p) > 1 else 0.0,
                               float(p[2]) if len(p) > 2 else 0.0)
        kind_id = KINDS[kind] if isinstance(kind, str) else int(kind)
        xs = cs = None
        on_dev = 0
        if device_ptrs is not None:
            xp, cp = device_ptrs
            on_dev = 1
            if n_obs is None:
                raise ValueError("n_obs is required with device pointers")
        else:
            xs = f8(x if x is not None else [])
            cs = None if choice is None else np.ascontiguousarray(choice, dtype=np.int32)
            xp = xs.ctypes.data
            cp = cs.ctypes.data if cs is not None else None
            if kind in ("mvnormal", "mvnormal_full"):
                n_obs, n_dim = xs.shape
            elif kind == "hier_normal":
                n_dim, n_per = xs.shape
                n_obs = n_dim * n_per
            elif kind == "binomial":
                n_obs = 1
            elif kind == "rastrigin":
                n_obs = 0
            elif kind in ("custom", "simulated"):
                if x is None:
                    n_obs, n_cols = 0, 0
                elif xs.ndim == 1:
                    n_obs, n_cols = xs.shape[0], 1
                elif xs.ndim == 2:
                    n_obs, n_cols = xs.shape
                else:
                    raise ValueError(f"{kind} data must be a vector or an n_obs x n_cols matrix")
            else:
                n_obs = xs.shape[0]
                if kind in ("lnr", "lba") and not n_dim:
                    n_dim = d - 1 if kind == "lnr" else d - 3
        sg = None if sigma is None else f8(sigma)
        cen = None if center is None else f8(center).reshape(-1)
        if cen is not None and cen.size != int(n_dim):
            raise ValueError(f"center needs {n_dim} entries")
        cv = None if cov is None else f8(cov)
        if kind == "mvnormal_full" and (cv is None or cv.shape != (int(n_dim), int(n_dim))):
            raise ValueError("mvnormal_full needs cov of shape (n_dim, n_dim)")
        src = None if source is None else source.encode() if isinstance(source, str) else bytes(source)
        m = _ffi.Model(kind_id, d, int(n_obs), int(n_dim), int(n_per), xp, cp, ptr(sg, _dp), float(lba_floor), pr, on_dev,
                       int(n_cols or 0), ptr(cv, _dp), ptr(cen, _dp), src, int(n_sim), float(sim_floor))
        self._keep = [xs, cs, sg, pr, cen, cv, src]
        check(_ffi.lib().demcmc_set_model(self._h, C.byref(m)))
        self.n_obs = int(n_obs)
        self.n_cols, self.n_sim = int(n_cols or 0), int(n_sim)

    # ---- state ---------------------------------------------------------------------------------
    def set_history(self, rows):
        """initialize_samples (utilities.jl:29-41): rows[n_initial][P][d], row i = the i-th sample_prior()
        draw of every particle id."""
        r = f8(rows).reshape(self.n_initial, -1, self.d)     # P of the handle, or P of the whole job when sharded
        check(_ffi.lib().demcmc_set_history(self._h, ptr(r, _dp)))

    def set_state(self, theta=None, ids=None):
        """theta=None after set_history: init_particle starts from samples[1, :, id] (utilities.jl:15)."""
        th = None if theta is None else f8(theta).reshape(self.P, self.d)
        idv = None if ids is None else np.ascontiguousarray(ids, dtype=np.int32)
        check(_ffi.lib().demcmc_set_state(self._h, ptr(th, _dp), ptr(idv, _ip)))

    def get_state(self):
        th = np.zeros((self.P, self.d))
        w = np.zeros(self.P)
        ids = np.zeros(self.P, dtype=np.int32)
        check(_ffi.lib().demcmc_get_state(self._h, ptr(th, _dp), ptr(w, _dp), ptr(ids, _ip)))
        return th, w, ids

    # ---- run -----------------------------------------------------------------------------------
    def run(self, n_iter):
        check(_ffi.lib().demcmc_run(self._h, int(n_iter)))
        self.iterations += n_iter
        self._last_iters = n_iter

    def replay(self, tape: dict, n_iter):
        """`tape`: dict of numpy arrays named after the demcmc_tape fields, whole-job shapes."""
        def get(name, dt):
            a = tape.get(name)
            if a is None:
                return None
            a = np.ascontiguousarray(a, dtype=dt)
            keep.append(a)
            return a
        keep = []
        t = _ffi.Tape(ptr(get("mig_u", "f8"), _dp), ptr(get("mig_n", "i4"), _ip), ptr(get("mig_groups", "i4"), _ip),
                      ptr(get("mig_pick_u", "f8"), _dp), ptr(get("kind", "u1"), _bp), ptr(get("idx", "i4"), _ip),
                      ptr(get("gamma1", "f8"), _dp), ptr(get("gamma2", "f8"), _dp), ptr(get("u_acc", "f8"), _dp),
                      ptr(get("noise", "f8"), _dp), ptr(get("keep", "u1"), _bp), ptr(get("idx_row", "i4"), _ip))
        check(_ffi.lib().demcmc_replay(self._h, C.byref(t), int(n_iter)))
        self.iterations += n_iter
        self._last_iters = n_iter

    # ---- results -------------------------------------------------------------------------------
    @property
    def n_rows(self):
        """rows of de.samples held: the n_initial prior rows + every store_every-th iteration"""
        return self.iterations // self.store_every + self.n_initial

    @property
    def stored_iterations(self):
        return self.iterations // self.store_every

    def samples(self):
        """de.samples in Julia memory order: returned as a numpy array of shape (P, d, n_rows),
        i.e. samples[id, k, row] == Julia samples[row+1, k+1, id+1]."""
        out = np.zeros((self.P, self.d, self.n_rows))
        check(_ffi.lib().demcmc_get_samples(self._h, ptr(out, _dp), self.n_rows))
        return out

    def accept(self):
        out = np.zeros((self.P, self.n_rows), dtype=np.uint8)
        check(_ffi.lib().demcmc_get_accept(self._h, ptr(out, _bp), self.n_rows))
        return out

    def lp(self):
        out = np.zeros((self.P, self.n_rows))
        check(_ffi.lib().demcmc_get_lp(self._h, ptr(out, _dp), self.n_rows))
        return out

    def chains(self, row0=0, n_rows=None):
        """bundle_samples on the device: array of shape (P, d+2, n_rows) in Julia memory order, i.e.
        out[c, k, r] == Julia Array(n_rows, d+2, P)[r+1, k+1, c+1] of iterations row0+r."""
        n = self.stored_iterations - row0 if n_rows is None else n_rows
        out = _out_empty((self.P, self.d + 2, max(n, 0)))
        if n > 0:
            check(_ffi.lib().demcmc_get_chains(self._h, int(row0), int(n), ptr(out, _dp)))
        return out

    def set_blocking_schedule(self, on):
        """blocking_on(de) per iteration (0-based from the chain's first iteration); beyond it: blocked."""
        a = np.ascontiguousarray(on, dtype=np.uint8).reshape(-1)
        check(_ffi.lib().demcmc_set_blocking_schedule(self._h, ptr(a, _bp), a.size))

    def set_weights(self, w):
        """The weights the saved particles carried (get_state()[1]); after set_state."""
        check(_ffi.lib().demcmc_set_weights(self._h, ptr(f8(w).reshape(self.P), _dp)))

    def set_iteration(self, iterations_done):
        """Resume: this handle continues a chain that already ran `iterations_done` iterations elsewhere
        (set_state with the saved theta and ids first or after; before the first run)."""
        check(_ffi.lib().demcmc_set_iteration(self._h, int(iterations_done)))

    def moments(self, row0=0, n_rows=None):
        """Pooled posterior summary computed on the device (no download of the draws): (count, mean[d],
        var[d] with ddof=1) over history rows [row0, row0+n_rows) and all local particles.  Rows count from the
        first history row, the n_initial prior rows included (as in samples() and diagnostics()); by default
        every stored row from row0 on."""
        n = self.n_rows - row0 if n_rows is None else n_rows
        cnt = C.c_int64(0)
        mean, m2 = np.zeros(self.d), np.zeros(self.d)
        check(_ffi.lib().demcmc_get_moments(self._h, int(row0), int(n), C.byref(cnt), ptr(mean, _dp), ptr(m2, _dp)))
        return cnt.value, mean, m2 / max(cnt.value - 1, 1)

    def diagnostics(self, row0=0, n_rows=None):
        """(split-R-hat[d], ESS[d]) of history rows [row0, row0+n_rows) computed on the device, every particle id one
        chain (demcmc_get_diagnostics): no download of the draws."""
        n = self.n_rows - row0 if n_rows is None else n_rows
        rhat, ess = np.zeros(self.d), np.zeros(self.d)
        check(_ffi.lib().demcmc_get_diagnostics(self._h, int(row0), int(n), ptr(rhat, _dp), ptr(ess, _dp)))
        return rhat, ess

    def history_by_slot(self, row0=0, n_rows=None):
        n = self.stored_iterations - row0 if n_rows is None else n_rows
        th = np.zeros((n, self.P, self.d))
        w = np.zeros((n, self.P))
        ids = np.zeros((n, self.P), dtype=np.int32)
        acc = np.zeros((n, self.P), dtype=np.uint8)
        check(_ffi.lib().demcmc_get_history_by_slot(self._h, row0, n, ptr(th, _dp), ptr(w, _dp), ptr(ids, _ip), ptr(acc, _bp)))
        return th, w, ids, acc

    def trace(self):
        S = self._last_iters * self.B
        out = {"prop_theta": np.zeros((S, self.P, self.d)), "prop_weight": np.zeros((S, self.P)),
               "log_adj": np.zeros((S, self.P)), "accepted": np.zeros((S, self.P), dtype=np.uint8)}
        check(_ffi.lib().demcmc_get_trace(self._h, ptr(out["prop_theta"], _dp), ptr(out["prop_weight"], _dp),
                                          ptr(out["log_adj"], _dp), ptr(out["accepted"], _bp)))
        return out

    def trace_xdot(self):
        """mvnormal / hier_normal: the cross term B the streamed likelihood kernel produced for every proposal
        of the last call, [S][P] (demcmc_get_trace_xdot)."""
        out = np.zeros((self._last_iters * self.B, self.P))
        check(_ffi.lib().demcmc_get_trace_xdot(self._h, ptr(out, _dp)))
        return out

    def eval_xdot(self, theta):
        th = f8(theta).reshape(-1, self.d)
        out = np.zeros(th.shape[0])
        check(_ffi.lib().demcmc_eval_xdot(self._h, ptr(th, _dp), th.shape[0], ptr(out, _dp)))
        return out

    def set_sufficient_stat(self, on=True):
        """Skip the O(N d) stream of the mvnormal / hier_normal likelihood (its cross term is analytically zero
        with mean-centred data); reported separately by bench.py, off by default."""
        check(_ffi.lib().demcmc_set_sufficient_stat(self._h, int(bool(on))))

    def migration_slots(self):
        out = np.full((max(1, self._last_iters), self.n_groups), -1, dtype=np.int32)
        check(_ffi.lib().demcmc_get_migration(self._h, ptr(out, _ip)))
        return out[: self._last_iters]

    def counters(self):
        c = _ffi.Counters()
        check(_ffi.lib().demcmc_get_counters(self._h, C.byref(c)))
        return {n: getattr(c, n) for n, _ in _ffi.Counters._fields_}

    def set_timing(self, l2_flush_bytes=0, time_loglik=False):
        check(_ffi.lib().demcmc_set_timing(self._h, int(l2_flush_bytes), int(bool(time_loglik))))

    def set_max_chunk(self, n_sweeps):
        check(_ffi.lib().demcmc_set_max_chunk(self._h, int(n_sweeps)))

    def set_lanes(self, n_lanes):
        check(_ffi.lib().demcmc_set_lanes(self._h, int(n_lanes)))

    def eval(self, theta):
        th = f8(theta).reshape(-1, self.d)
        n = th.shape[0]
        ll = np.zeros(n)
        pr = np.zeros(n)
        check(_ffi.lib().demcmc_eval(self._h, ptr(th, _dp), n, ptr(ll, _dp), ptr(pr, _dp)))
        return ll, pr

    def eval_simulated(self, theta, sweep, unit, sims=False):
        """Test hook of a simulated model (demcmc_eval_simulated): the log-likelihoods of theta[n][d] under the explicit
        simulation keys (sweep[i], unit[i]), and with sims=True also the simulations, an array [n, n_sim, n_cols]."""
        th = f8(theta).reshape(-1, self.d)
        n = th.shape[0]
        sw = np.ascontiguousarray(np.broadcast_to(np.asarray(sweep, dtype=np.uint32), (n,)))
        un = np.ascontiguousarray(np.broadcast_to(np.asarray(unit, dtype=np.uint32), (n,)))
        ll = np.zeros(n)
        out = np.zeros((n, self.n_sim, self.n_cols)) if sims else None
        u32 = C.POINTER(C.c_uint32)
        check(_ffi.lib().demcmc_eval_simulated(self._h, ptr(th, _dp), n, ptr(sw, u32), ptr(un, u32), ptr(ll, _dp), ptr(out, _dp)))
        return (ll, out) if sims else ll

    def eval_pointwise(self, theta, obs0=0, n_obs=None):
        """log p(y_i | theta_s) for the draws theta[n][d] and observations [obs0, obs0 + n_obs) of the bound model (all from
        obs0 by default): an array [n, n_obs] (demcmc_eval_pointwise; priors are left out)."""
        th = f8(theta).reshape(-1, self.d)
        n_obs = self.n_obs - obs0 if n_obs is None else int(n_obs)
        out = np.empty((th.shape[0], max(n_obs, 0)))
        check(_ffi.lib().demcmc_eval_pointwise(self._h, ptr(th, _dp), th.shape[0], int(obs0), n_obs, ptr(out, _dp)))
        return out

    def loo(self, theta):
        """PSIS-LOO and WAIC of every observation over the draws theta[n][d] (demcmc_loo, 2 <= n <= 16384): the arrays
        (elpd_loo, pareto_k, lppd, p_waic), each [n_obs]."""
        th = f8(theta).reshape(-1, self.d)
        out = [np.empty(self.n_obs) for _ in range(4)]
        check(_ffi.lib().demcmc_loo(self._h, ptr(th, _dp), th.shape[0], *(ptr(a, _dp) for a in out)))
        return tuple(out)

    # ---- power posteriors ----------------------------------------------------------------------
    def set_temperatures(self, t):
        """Temper every group of the job: t[n_groups] in [0, 1]; a group's weights become prior + t * loglike
        (demcmc_set_temperatures).  After set_model, before set_state."""
        a = f8(t).reshape(-1)
        self._temperatures = a
        check(_ffi.lib().demcmc_set_temperatures(self._h, ptr(a, _dp), a.size))

    def loglike(self):
        """The stored untempered log-likelihoods of a tempered handle, in the layout of lp(): shape (P, n_rows); the
        n_initial prior rows are NaN (demcmc_get_loglike)."""
        out = np.zeros((self.P, self.n_rows))
        check(_ffi.lib().demcmc_get_loglike(self._h, ptr(out, _dp), self.n_rows))
        return out

    def power_posterior(self, row0=None, n_rows=None):
        """Thermodynamic-integration and stepping-stone estimates of log p(y) over the stored rows [row0, row0 + n_rows)
        (by default every row after the n_initial prior rows) of the rungs of a tempered handle (demcmc_power_posterior):
        a dict of the totals and the per-rung arrays t, mean_ll, var_ll, ess_ll, rhat_ll, log_ratio."""
        row0 = self.n_initial if row0 is None else int(row0)
        n = self.n_rows - row0 if n_rows is None else int(n_rows)
        cap = self.n_groups
        ev = _ffi.Evidence()
        arr = {k: np.zeros(cap) for k in ("t", "mean_ll", "var_ll", "ess_ll", "rhat_ll", "log_ratio")}
        check(_ffi.lib().demcmc_power_posterior(self._h, row0, n, cap, C.byref(ev), *(ptr(arr[k], _dp) for k in
                                                ("t", "mean_ll", "var_ll", "ess_ll", "rhat_ll", "log_ratio"))))
        out = {k: getattr(ev, k) for k, _ in _ffi.Evidence._fields_}
        out.update({k: v[: ev.n_rungs] for k, v in arr.items()})
        return out

    def comm_init(self, uid: bytes, rank: int, n_ranks: int):
        buf = np.frombuffer(uid, dtype=np.uint8).copy()
        check(_ffi.lib().demcmc_comm_init(self._h, ptr(buf, _bp), rank, n_ranks))


def compile_loglike(source):
    """Compiles a custom likelihood source for sm_100a (demcmc_compile_loglike; no device needed).  Raises DemcmcError
    with the compiler log when it does not compile; the result is cached for later set_model calls."""
    src = source.encode() if isinstance(source, str) else bytes(source)
    log = C.create_string_buffer(1 << 16)
    rc = _ffi.lib().demcmc_compile_loglike(src, log, len(log))
    if rc != 0:
        raise _ffi.DemcmcError(rc, log.value.decode(errors="replace") or _ffi.lib().demcmc_last_error().decode(errors="replace"))


def compile_simulator(source):
    """Compiles a simulated-likelihood source (DEMCMC_SIMULATED) for sm_100a (demcmc_compile_simulator; no device needed).
    Raises DemcmcError with the compiler log when it does not compile; the result is cached for later set_model calls."""
    src = source.encode() if isinstance(source, str) else bytes(source)
    log = C.create_string_buffer(1 << 16)
    rc = _ffi.lib().demcmc_compile_simulator(src, log, len(log))
    if rc != 0:
        raise _ffi.DemcmcError(rc, log.value.decode(errors="replace") or _ffi.lib().demcmc_last_error().decode(errors="replace"))


def comm_unique_id() -> bytes:
    buf = np.zeros(128, dtype=np.uint8)
    check(_ffi.lib().demcmc_comm_unique_id(ptr(buf, _bp)))
    return buf.tobytes()


# ---- particle algebra (known-answer tests) ------------------------------------------------------
def op_project(p1, p2, device=0):
    p1, p2 = f8(p1), f8(p2)
    out = np.zeros_like(p1)
    check(_ffi.lib().demcmc_op_project(device, ptr(p1, _dp), ptr(p2, _dp), p1.size, ptr(out, _dp)))
    return out


def op_reset(prop, pt, mask, device=0):
    prop, pt = f8(prop), f8(pt)
    mask = np.ascontiguousarray(mask, dtype=np.uint8)
    out = np.zeros_like(prop)
    check(_ffi.lib().demcmc_op_reset(device, ptr(prop, _dp), ptr(pt, _dp), ptr(mask, _bp), prop.size, ptr(out, _dp)))
    return out


def op_de_proposal(pt, pm, pn, pb, g1, g2, b, device=0):
    pt, pm, pn, b = f8(pt), f8(pm), f8(pn), f8(b)
    pbv = None if pb is None else f8(pb)
    out = np.zeros_like(pt)
    check(_ffi.lib().demcmc_op_de_proposal(device, ptr(pt, _dp), ptr(pm, _dp), ptr(pn, _dp), ptr(pbv, _dp), g1, g2,
                                           ptr(b, _dp), pt.size, ptr(out, _dp)))
    return out


def op_snooker(pt, pz, pm, pn, g, b, device=0):
    pt, pz, pm, pn, b = f8(pt), f8(pz), f8(pm), f8(pn), f8(b)
    out = np.zeros_like(pt)
    adj = np.zeros(1)
    check(_ffi.lib().demcmc_op_snooker(device, ptr(pt, _dp), ptr(pz, _dp), ptr(pm, _dp), ptr(pn, _dp), g, ptr(b, _dp),
                                       pt.size, ptr(out, _dp), ptr(adj, _dp)))
    return out, float(adj[0])


def op_accept(w_prop, w_cur, log_adj, u, device=0):
    a, b, c, d = f8(w_prop), f8(w_cur), f8(log_adj), f8(u)
    out = np.zeros(a.size, dtype=np.uint8)
    check(_ffi.lib().demcmc_op_accept(device, ptr(a, _dp), ptr(b, _dp), ptr(c, _dp), ptr(d, _dp), a.size, ptr(out, _bp)))
    return out.astype(bool)


def op_select(w, u, device=0):
    w = f8(w)
    o = np.zeros(2, dtype=np.int32)
    check(_ffi.lib().demcmc_op_select(device, ptr(w, _dp), w.size, u, o[:1].ctypes.data_as(_ip), o[1:].ctypes.data_as(_ip)))
    return int(o[0]), int(o[1])


def fp64_peak(device=0):
    v = np.zeros(1)
    check(_ffi.lib().demcmc_fp64_peak(device, ptr(v, _dp)))
    return float(v[0])


def fp64_peaks(device=0):
    """(DFMA loop, DMMA m8n8k4 loop) in TFLOP/s; one pipe on B200, the larger is the roofline."""
    a, b = np.zeros(1), np.zeros(1)
    check(_ffi.lib().demcmc_fp64_peaks(device, ptr(a, _dp), ptr(b, _dp)))
    return float(a[0]), float(b[0])


def copy_peak(device=0):
    v = np.zeros(1)
    check(_ffi.lib().demcmc_copy_peak(device, ptr(v, _dp)))
    return float(v[0])

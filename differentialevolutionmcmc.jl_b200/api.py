"""Host-side mirror of the reference's interface for the population-step path.

Same names, argument meaning and error behaviour as DifferentialEvolutionMCMC.jl:
`DEModel(; prior_loglike, loglike, names, sample_prior, data)` (src/structs.jl:176-189),
`DE(; n_groups, Np, burnin, ..., bounds, sample_prior)` (src/structs.jl:80-131) and
`sample(model, de, n_iter)` / `sample(model, de, MCMCThreads(), n_iter)` (src/main.jl:19-71).
The one new type is `GPULoglike`, which binds the model to a registered hand-written kernel; a
plain callable raises instead of falling back to the CPU.  The Julia version of this file is
julia/GPULoglike.jl (same ABI calls, not executable in this image).
"""
from __future__ import annotations

import numpy as np

from .handle import Handle, compile_loglike, compile_simulator


# ---- registered priors (replace prior_loglike closures) -----------------------------------------
class _PriorSpec:
    kind = "flat"
    a = 0.0
    b = 0.0
    ref = None

    def logpdf_note(self):
        return self.kind


class Flat(_PriorSpec):
    pass


class Normal(_PriorSpec):
    """Normal(mu, sd) -- Distributions.Normal"""
    kind = "normal"

    def __init__(self, mu=0.0, sd=1.0):
        self.a, self.b = float(mu), float(sd)


class HalfCauchy(_PriorSpec):
    """truncated(Cauchy(loc, scale), 0, Inf)"""
    kind = "halfcauchy"

    def __init__(self, loc=0.0, scale=1.0):
        self.a, self.b = float(loc), float(scale)


class Uniform(_PriorSpec):
    kind = "uniform"

    def __init__(self, a, b):
        self.a, self.b = float(a), float(b)


class Beta(_PriorSpec):
    kind = "beta"

    def __init__(self, a=1.0, b=1.0):
        self.a, self.b = float(a), float(b)


class NormalRef(_PriorSpec):
    """Normal(mean, sd = another (scalar) named parameter): the hierarchical prior
    sum(logpdf.(Normal(0, σβ0), β0)) of Examples/Hierarchical_Example.jl:30."""
    kind = "normal_ref"

    def __init__(self, mean, sd):
        self.a, self.ref = float(mean), sd


class GPUPrior:
    """One registered prior spec per NAMED parameter, applied to every element of an array
    parameter.  Replaces `prior_loglike(θ...)`."""

    def __init__(self, *specs):
        if len(specs) == 1 and isinstance(specs[0], (list, tuple)):
            specs = tuple(specs[0])
        for s in specs:
            if not isinstance(s, _PriorSpec):
                raise TypeError(f"{s!r} is not a registered prior spec (Normal, HalfCauchy, Uniform, Beta, NormalRef, Flat)")
        self.specs = specs


class GPULoglike:
    """Binds a model to a registered hand-written likelihood kernel.

    GPULoglike("gaussian", x)                    sum(logpdf.(Normal(μ,σ), x))
    GPULoglike("mvnormal", X)                    X is n_obs × n_dim; sum(logpdf(MvNormal(μ, σ²I), X'))
    GPULoglike("binomial", N=10, k=3)            logpdf(Binomial(N,θ), k)
    GPULoglike("lnr", choice=c, rt=t)            sum(logpdf(LNR(;ν,τ), data)), σ = 1 unless sigma=...
    GPULoglike("lba", choice=c, rt=t)            sum(logpdf.(LBA(;ν,A,k,τ), c, t))
    GPULoglike("hier_normal", Y)                 Y is n_subj × n_per (Examples/Hierarchical_Example.jl)
    GPULoglike("mvnormal_full", X, cov=Σ)        sum(logpdf(MvNormal(μ, σ²Σ), X')) with a known covariance Σ
    GPULoglike("custom", X, source=src)          sum_i demcmc_obs(par, X[i]) + demcmc_particle(θ): a likelihood written as
                                                 CUDA C++ (include/demcmc_b200.h: DEMCMC_CUSTOM), compiled here for
                                                 sm_100a; X is a vector, an n_obs × n_cols matrix, or None (no data)
    GPULoglike("simulated", X, source=src, n_sim=M, floor=1e-10)
                                                 a likelihood estimated from M simulations per proposal of the CUDA C++
                                                 simulator demcmc_simulate (include/demcmc_b200.h: DEMCMC_SIMULATED): a
                                                 Gaussian kernel density per label; X is a vector of values or an n_obs × 2
                                                 matrix of (label 1..8, value) rows
    (Examples/Guassian_Example_Vector.jl is the "gaussian" kernel: its loglike(data, θ...) destructures μ, σ)
    """
    KINDS = ("gaussian", "mvnormal", "binomial", "lnr", "lba", "hier_normal", "rastrigin", "mvnormal_full", "custom", "simulated")

    def __init__(self, kind, x=None, *, choice=None, rt=None, N=None, k=None, sigma=None, lba_floor=1e-10, cov=None,
                 source=None, n_sim=None, floor=1e-10):
        kind = str(kind).lstrip(":")
        if kind not in self.KINDS:
            raise ValueError(f"no registered kernel for {kind!r}; registered: {self.KINDS}")
        self.kind = kind
        self.choice = None
        self.sigma = sigma
        self.lba_floor = lba_floor
        self.cov = None if cov is None else np.ascontiguousarray(cov, dtype=np.float64)   # mvnormal_full: the known covariance
        self.source = None
        self.n_sim, self.sim_floor = 0, 1e-10
        if kind == "simulated":
            if not isinstance(source, (str, bytes)) or not source:
                raise ValueError("simulated needs source=: CUDA C++ text that defines demcmc_simulate (include/demcmc_b200.h)")
            if x is None:
                raise ValueError("simulated needs data: a vector of values or an n_obs x 2 matrix of (label, value) rows")
            self.x = np.ascontiguousarray(x, dtype=np.float64)
            if self.x.ndim not in (1, 2) or (self.x.ndim == 2 and self.x.shape[1] not in (1, 2)):
                raise ValueError("simulated data must be a vector (n_cols = 1) or an n_obs x 2 matrix of (label, value) rows (n_cols = 2)")
            if self.x.shape[0] < 1:
                raise ValueError("simulated data need at least one observation")
            vals = self.x if self.x.ndim == 1 else self.x[:, -1]
            if not np.all(np.isfinite(vals)):
                raise ValueError("simulated data values must be finite")
            if self.x.ndim == 2 and self.x.shape[1] == 2:
                lab = self.x[:, 0]
                if not np.all((lab == np.floor(lab)) & (lab >= 1) & (lab <= 8)):
                    raise ValueError("simulated data labels must be integers in 1..8")
            if n_sim is None or not 16 <= int(n_sim) <= 16384:
                raise ValueError(f"simulated needs n_sim in [16, 16384] simulations per proposal, got {n_sim}")
            if not float(floor) > 0.0:
                raise ValueError(f"simulated needs floor > 0, got {floor}")
            compile_simulator(source)        # a source that does not compile fails here, with the compiler log
            self.source, self.n_sim, self.sim_floor = source, int(n_sim), float(floor)
        elif kind == "custom":
            if not isinstance(source, (str, bytes)) or not source:
                raise ValueError("custom needs source=: CUDA C++ text that defines demcmc_obs (include/demcmc_b200.h)")
            self.x = None if x is None else np.ascontiguousarray(x, dtype=np.float64)
            if self.x is not None and (self.x.ndim not in (1, 2) or (self.x.ndim == 2 and self.x.shape[1] == 0)):
                raise ValueError("custom data must be a vector or an n_obs x n_cols matrix with n_cols >= 1")
            compile_loglike(source)          # a source that does not compile fails here, with the compiler log
            self.source = source
        elif kind == "rastrigin":              # the objective of test/optimization_tests.jl:15-23: no data
            self.x = np.zeros(0)
        elif kind == "binomial":
            if N is None or k is None:
                raise ValueError("binomial needs N and k")
            self.x = np.array([float(N), float(k)])
        elif kind in ("lnr", "lba"):
            if choice is None or rt is None:
                raise ValueError(f"{kind} needs choice and rt")
            self.x = np.ascontiguousarray(rt, dtype=np.float64)
            self.choice = np.ascontiguousarray(choice, dtype=np.int32)
            if self.x.shape != self.choice.shape or self.x.ndim != 1:
                raise ValueError("choice and rt must be vectors of the same length")
        else:
            if x is None:
                raise ValueError(f"{kind} needs data")
            self.x = np.ascontiguousarray(x, dtype=np.float64)
            if kind in ("mvnormal", "hier_normal", "mvnormal_full") and self.x.ndim != 2:
                raise ValueError(f"{kind} data must be a matrix")

    def __call__(self, *a, **k):
        raise TypeError("GPULoglike is evaluated on the device; it is not a host callable")


class MCMCThreads:
    """Marker mirroring AbstractMCMC.MCMCThreads(): the reference runs one task per group
    (src/main.jl:135-148); on the device every group is always updated concurrently."""


def resample(*a):
    """DE(sample=resample): DE-MCz donors from the history (src/crossover.jl:113-124)."""
    raise TypeError("resample is a donor selector for DE(sample=...), not a host function")


def maximize(*a):
    """DE(update_particle=maximize): the greedy maximize! of optimize (src/utilities.jl:212-218)."""
    raise TypeError("maximize is an update selector for DE(update_particle=...), not a host function")


def minimize(*a):
    """DE(update_particle=minimize): minimize! (src/utilities.jl:220-226)."""
    raise TypeError("minimize is an update selector")


def mh_update(*a):
    raise TypeError("mh_update is an update selector")


def evaluate_fun(*a):
    """DE(evaluate_fitness=evaluate_fun): the registered kernel alone, no prior (src/utilities.jl:113-120)."""
    raise TypeError("evaluate_fun is a fitness selector")


def compute_posterior(*a):
    raise TypeError("compute_posterior is a fitness selector")


def random_gamma(*a):
    raise TypeError("random_gamma is a proposal selector for DE(generate_proposal=...), not a host function")


def fixed_gamma(*a):
    raise TypeError("fixed_gamma is a proposal selector")


def variable_gamma(*a):
    raise TypeError("variable_gamma is a proposal selector")


_PROPOSAL_NAMES = {random_gamma: "random_gamma", fixed_gamma: "fixed_gamma", variable_gamma: "variable_gamma"}


class DEModel:
    """DEModel(; prior_loglike, loglike, names, sample_prior, data=nothing) (src/structs.jl:176-189)."""

    def __init__(self, *args, prior_loglike=None, loglike, names, sample_prior, data=None, **kwargs):
        if args or kwargs:
            raise TypeError("extra loglike arguments only make sense for host closures, which the B200 path does not run")
        self.prior_loglike = prior_loglike
        self.loglike = loglike
        self.sample_prior = sample_prior
        self.names = tuple(names)
        self.data = data


def GPUDEModel(*, prior_loglike=None, loglike, names, sample_prior):
    """The GPU model's own constructor of julia/GPULoglike.jl (there the package's keyword constructor DEModel(args...; ...)
    must stay untouched for CPU models); here simply DEModel."""
    return DEModel(prior_loglike=prior_loglike, loglike=loglike, names=names, sample_prior=sample_prior)


class DE:
    """DE(; n_groups=4, Np, burnin=1000, discard_burnin=true, α=.1, β=.1, ϵ=.001, σ=.05, κ=1.0,
    θsnooker=0.0, bounds, n_initial=0, generate_proposal=random_gamma, blocking_on=x->false,
    blocks=[false], sample_prior) (src/structs.jl:80-131).  Greek keywords are accepted as in
    Julia; ASCII aliases alpha, beta, eps, sigma, kappa, theta_snooker too."""

    def __init__(self, *, n_groups=4, priors=None, Np, burnin=1000, discard_burnin=True, bounds, n_initial=0,
                 generate_proposal=random_gamma, update_particle=None, evaluate_fitness=None, sample=None,
                 blocking_on=None, blocks=None, sample_prior, seed=None, **greek):
        alias = {"α": "alpha", "β": "beta", "ϵ": "eps", "ε": "eps", "σ": "sigma", "κ": "kappa", "θsnooker": "theta_snooker"}
        vals = {"alpha": 0.1, "beta": 0.1, "eps": 0.001, "sigma": 0.05, "kappa": 1.0, "theta_snooker": 0.0}
        for k, v in greek.items():
            k2 = alias.get(k, k)
            if k2 not in vals:
                raise TypeError(f"DE() got an unexpected keyword argument {k!r}")
            vals[k2] = float(v)
        if n_groups == 1 and vals["alpha"] > 0:
            vals["alpha"] = 0.0   # structs.jl:102-105 (the reference warns)
        self.n_groups, self.Np, self.burnin, self.discard_burnin = int(n_groups), int(Np), int(burnin), bool(discard_burnin)
        self.α, self.β, self.ϵ, self.σ, self.κ, self.θsnooker = (vals[k] for k in ("alpha", "beta", "eps", "sigma", "kappa", "theta_snooker"))
        self.bounds = tuple(bounds)
        self.n_initial = int(n_initial)
        self.iter = 1
        if update_particle not in (None, mh_update, maximize, minimize):
            raise TypeError("update_particle must be mh_update, maximize or minimize: a custom host function cannot run on the device")
        if evaluate_fitness not in (None, compute_posterior, evaluate_fun):
            raise TypeError("evaluate_fitness must be compute_posterior or evaluate_fun")
        self.update_particle = update_particle or mh_update
        self.evaluate_fitness = evaluate_fitness or compute_posterior
        if sample is not None and sample is not resample:
            raise TypeError("sample must be left at its default (donors from the current group) or be `resample`: a custom host function cannot run on the device")
        self.sample = sample
        if sample is resample and self.n_initial * self.n_groups * self.Np < 3:
            raise ValueError("sample = resample draws donors from rows 1:de.iter-1 of de.samples: it needs n_initial > 0")
        if generate_proposal not in _PROPOSAL_NAMES:
            raise TypeError("generate_proposal must be random_gamma, fixed_gamma or variable_gamma: a custom host function cannot run on the device")
        self.generate_proposal = generate_proposal
        self.blocking_on = blocking_on if blocking_on is not None else (lambda de: False)
        self.blocks = blocks if blocks is not None else [False]
        self.sample_prior = sample_prior
        self.seed = seed
        self.samples = None

    # ASCII views
    alpha = property(lambda s: s.α)
    beta = property(lambda s: s.β)
    eps = property(lambda s: s.ϵ)
    sigma = property(lambda s: s.σ)
    kappa = property(lambda s: s.κ)
    theta_snooker = property(lambda s: s.θsnooker)


class Chains:
    """Minimal stand-in for MCMCChains.Chains as produced by bundle_samples (src/main.jl:222-250):
    value[Ns, n_flat_parms + 2, n_chains] with the internals "acceptance" and "lp" last."""

    def __init__(self, value, names, parameters):
        self.value = value
        self.names = list(names)
        self.parameters = list(parameters)
        self.internals = ["acceptance", "lp"]

    def __len__(self):
        return self.value.shape[0]

    def _par(self):
        return self.value[:, : len(self.names) - 2, :]

    def mean(self):
        return self._par().mean(axis=(0, 2))

    def std(self):
        v = self._par()
        return v.transpose(1, 0, 2).reshape(v.shape[1], -1).std(axis=1, ddof=1)

    def rhat(self):
        from .diagnostics import split_rhat
        v = self._par()
        return np.array([split_rhat(v[:, k, :]) for k in range(v.shape[1])])

    def ess(self):
        from .diagnostics import bulk_ess
        v = self._par()
        return np.array([bulk_ess(v[:, k, :]) for k in range(v.shape[1])])

    def describe(self):
        return {"parameters": self.names[:-2], "mean": self.mean(), "std": self.std(), "rhat": self.rhat(), "ess": self.ess()}


# ---- flattening helpers (get_names, src/utilities.jl:131-149) -----------------------------------
def _shapes(theta0):
    return [np.shape(v) for v in theta0]


def _flatten(theta):
    out = []
    for v in theta:
        a = np.asarray(v, dtype=np.float64)
        out.extend(a.reshape(-1, order="F").tolist() if a.ndim else [float(a)])
    return out


def _fill_flat(theta, out):
    """_flatten straight into a row of the state matrix (the P sample_prior() calls of sample_init are the host-side
    cost of a short run: no lists in between)"""
    k = 0
    for v in theta:
        if isinstance(v, float):
            out[k] = v
            k += 1
        elif isinstance(v, np.ndarray) and v.ndim:
            n = v.size
            out[k:k + n] = v if v.ndim == 1 else v.reshape(-1, order="F")
            k += n
        elif np.ndim(v):
            a = np.asarray(v, dtype=np.float64)
            out[k:k + a.size] = a.reshape(-1, order="F")
            k += a.size
        else:
            out[k] = v
            k += 1


def _draw_states(sample_prior, n, d):
    out = np.empty((n, d))
    for p in range(n):
        _fill_flat(sample_prior(), out[p])
    return out


def _flat_names(names, shapes):
    out = []
    for n, sh in zip(names, shapes):
        if len(sh) == 0:
            out.append(str(n))
        else:
            for idx in np.ndindex(*sh[::-1]):
                out.append(f"{n}[{','.join(str(i + 1) for i in idx[::-1])}]")
    return out


def _expand(per_name, shapes, what):
    if len(per_name) < len(shapes):
        per_name = list(per_name) + [None] * (len(shapes) - len(per_name))   # zip truncation (utilities.jl:74)
    out = []
    for v, sh in zip(per_name, shapes):
        n = int(np.prod(sh)) if len(sh) else 1
        out.extend([v] * n)
    return out


def _expand_block(block, shapes):
    out = []
    for b, sh in zip(block, shapes):
        n = int(np.prod(sh)) if len(sh) else 1
        if np.ndim(b) == 0:
            out.extend([bool(b)] * n)
        else:
            a = np.asarray(b, dtype=bool)
            if a.size != n:
                raise ValueError("block mask shape does not match the parameter")
            out.extend(a.reshape(-1, order="F").tolist())
    return out


def _prior_table(model, shapes, needed=True):
    pl = model.prior_loglike
    if pl is None and not needed:          # evaluate_fun! never calls prior_loglike (utilities.jl:113-120)
        return [("flat", 0.0, 0.0, 0)] * sum(int(np.prod(sh)) if len(sh) else 1 for sh in shapes)
    if not isinstance(pl, GPUPrior):
        raise TypeError(
            "prior_loglike must be a GPUPrior of registered specs: a host closure would need a host round trip per "
            "particle and the B200 path never falls back to the CPU")
    if len(pl.specs) != len(shapes):
        raise ValueError(f"GPUPrior has {len(pl.specs)} specs for {len(shapes)} named parameters")
    starts, pos = {}, 0
    for n, sh in zip(model.names, shapes):
        starts[str(n)] = (pos, sh)
        pos += int(np.prod(sh)) if len(sh) else 1
    table = []
    for spec, sh in zip(pl.specs, shapes):
        n = int(np.prod(sh)) if len(sh) else 1
        ref = 0
        if spec.kind == "normal_ref":
            key = str(spec.ref).lstrip(":")
            if key not in starts or len(starts[key][1]) != 0:
                raise ValueError(f"NormalRef sd {spec.ref!r} must name a scalar parameter")
            ref = starts[key][0]
        table.extend([(spec.kind, spec.a, spec.b, ref)] * n)
    return table


def _blocking_schedule(de: DE, n_iter):
    """blocking_on(de) is a function of the sampler, evaluated once per iteration with de.iter = iter +
    n_initial (src/main.jl:34,137,162): evaluated here for the n_iter iterations to come."""
    keep = de.iter
    try:
        on = []
        for it in range(1, n_iter + 1):
            de.iter = it + de.n_initial
            on.append(bool(de.blocking_on(de)))
    finally:
        de.iter = keep
    return on


class _Background:
    """Runs one library call on a host thread (ctypes releases the GIL for its duration) while the caller goes on in
    Python: sample() uploads and packs the data set (demcmc_set_model, a few ms for tens of MB) while the P sample_prior()
    calls of sample_init run.  join() re-raises what the call raised."""

    def __init__(self, fn):
        import threading
        self.err = None

        def run():
            try:
                fn()
            except BaseException as e:      # noqa: BLE001  (re-raised by join)
                self.err = e
        self.t = threading.Thread(target=run)
        self.t.start()

    def join(self):
        self.t.join()
        if self.err is not None:
            raise self.err


def build_handle(model: DEModel, de: DE, device=0, trace=False, group_begin=0, group_count=0, n_iter=None, devices=None, store_every=1,
                 background_model=False):
    """background_model=True: demcmc_set_model runs on a host thread; the fourth return value must be join()ed before the
    handle is used."""
    """Everything `sample` does before the iteration loop; also used by bench.py and the tests."""
    ll = model.loglike
    if not isinstance(ll, GPULoglike):
        raise TypeError(
            "loglike must be a GPULoglike bound to a registered kernel "
            f"{GPULoglike.KINDS}; an arbitrary closure cannot run on the device and there is no CPU fallback "
            "(write the likelihood as CUDA source instead: GPULoglike(\"custom\", X, source=...))")
    theta0 = model.sample_prior()
    shapes = _shapes(theta0)
    d = len(_flatten(theta0))
    lo = [(-np.inf if b is None else float(b[0])) for b in _expand(list(de.bounds), shapes, "bounds")]
    hi = [(np.inf if b is None else float(b[1])) for b in _expand(list(de.bounds), shapes, "bounds")]
    blocks, schedule = None, None
    on = _blocking_schedule(de, n_iter) if n_iter is not None else [bool(de.blocking_on(de))]
    if any(on):
        blocks = np.array([_expand_block(b, shapes) for b in de.blocks], dtype=np.uint8)
        if not all(on):
            schedule = on                                   # block updating in some iterations only
    seed = de.seed if de.seed is not None else int(np.random.SeedSequence().generate_state(2, dtype=np.uint32).view(np.uint64)[0])
    h = Handle(de.n_groups, de.Np, d, lo, hi, burnin=de.burnin, n_initial=de.n_initial, alpha=de.α, beta=de.β, eps=de.ϵ,
               sigma=de.σ, kappa=de.κ, theta_snooker=de.θsnooker, proposal=_PROPOSAL_NAMES[de.generate_proposal],
               blocks=blocks, seed=seed, device=device, trace=trace, group_begin=group_begin, group_count=group_count,
               resample=de.sample is resample, update={mh_update: "mh", maximize: "maximize", minimize: "minimize"}[de.update_particle],
               fitness="fun" if de.evaluate_fitness is evaluate_fun else "posterior", blocking_schedule=schedule, devices=devices,
               store_every=store_every)
    table = _prior_table(model, shapes, needed=de.evaluate_fitness is not evaluate_fun)

    def bind():
        h.set_model(ll.kind, table, x=ll.x, choice=ll.choice, sigma=ll.sigma, lba_floor=ll.lba_floor, cov=ll.cov, source=ll.source,
                    n_sim=ll.n_sim, sim_floor=ll.sim_floor)
    if background_model:
        return h, shapes, d, _Background(bind)
    bind()
    return h, shapes, d


def _init_state(h, model: DEModel, de: DE, d, binding, temperatures=None):
    """The particles of sample_init, once the model is bound; temperatures (per group of the job) temper the handle first."""
    P = de.n_groups * de.Np
    rows = theta0 = None
    if de.n_initial > 0:
        # initialize_samples (src/utilities.jl:29-41): for every particle id, n_initial sample_prior()
        # draws; init_particle then starts each particle from samples[1, :, id] (utilities.jl:15)
        rows = np.empty((de.n_initial, P, d))
        for p in range(P):
            for i in range(de.n_initial):
                _fill_flat(model.sample_prior(), rows[i, p])
    else:
        # sample_init (src/main.jl:263-271): one sample_prior() per particle, id order -- drawn while the data upload runs
        theta0 = _draw_states(model.sample_prior, P, d)
    binding.join()                                       # the data set is on the device and packed
    if temperatures is not None:
        h.set_temperatures(temperatures)
    if rows is not None:
        h.set_history(rows)
    h.set_state(theta0)


def sample(model: DEModel, de: DE, *args, progress=False, device=0, devices=None, store_every=1, **kwargs):
    """sample(model, de, n_iter) / sample(model, de, MCMCThreads(), n_iter): runs all n_iter
    iterations on the device in ONE library call and returns the chains (src/main.jl:19-71).
    devices=[0, 1, ...]: the groups shard over several GPUs of the box from this one process (demcmc_config.n_devices).
    store_every=k: thinning -- the Chains hold iterations k, 2k, ... (burnin is then counted in kept rows: burnin // k)."""
    if len(args) == 2 and isinstance(args[0], MCMCThreads):
        n_iter = int(args[1])
    elif len(args) == 1:
        n_iter = int(args[0])
    else:
        raise TypeError("sample(model, de, n_iter) or sample(model, de, MCMCThreads(), n_iter)")
    h, shapes, d, binding = build_handle(model, de, device=device, n_iter=n_iter, devices=devices, store_every=store_every, background_model=True)
    try:
        _init_state(h, model, de, d, binding)
        h.run(n_iter)
        de.iter = n_iter + de.n_initial
        # bundle_samples (src/main.jl:222-250) runs on the device: one gather, one download, and the
        # host only wraps the array (Julia memory order) in a view
        offset = (de.burnin // h.store_every) if de.discard_burnin else 0
        arr = h.chains(offset, max(n_iter // h.store_every - offset, 0))
        de.samples = arr[:, :d, :]                       # what bundle_samples keeps of de.samples
        names = _flat_names(model.names, shapes) + ["acceptance", "lp"]
        return Chains(arr.transpose(2, 1, 0), names, [str(n) for n in model.names])
    finally:
        try:
            binding.join()                                   # (an exception above: let the upload finish before the handle goes)
        except BaseException:                                # noqa: BLE001
            pass
        h.close()


def power_posterior(model: DEModel, de: DE, n_iter, temperatures=None, n_temperatures=32, power=5.0, device=0, devices=None,
                    store_every=1):
    """The marginal likelihood log p(y) by power posteriors, in ONE run: rung k is de.n_groups groups of de.Np particles whose
    weights are prior + t_k loglike, t_k = (k / (K - 1))^power by default (Friel & Pettitt 2008), all K rungs in one handle of
    K * de.n_groups groups.  Burn-in is dropped as sample() drops it.  Returns a dict: the totals log_z_ti (trapezoid rule),
    log_z_ti2 (corrected trapezoid), log_z_ss (stepping stones) and their standard errors se_ti, se_ss; the per-rung arrays
    t, mean_ll, var_ll, ess_ll, rhat_ll, log_ratio (include/demcmc_b200.h: demcmc_power_posterior); and chains, the t = 1
    rung's Chains, a posterior sample like sample()'s."""
    import copy
    t = np.asarray([(k / (n_temperatures - 1)) ** power for k in range(n_temperatures)] if temperatures is None else temperatures, dtype=np.float64)
    K = t.size
    if de.α > 0 and K * de.n_groups > 1:
        raise ValueError("power_posterior runs every rung as groups of one handle, and migration would move particles between "
                         "temperatures: pass DE(α = 0)")
    job = copy.copy(de)
    job.n_groups = K * de.n_groups
    n_iter = int(n_iter)
    h, shapes, d, binding = build_handle(model, job, device=device, n_iter=n_iter, devices=devices, store_every=store_every, background_model=True)
    try:
        _init_state(h, model, job, d, binding, temperatures=np.repeat(t, de.n_groups))
        h.run(n_iter)
        offset = (de.burnin // h.store_every) if de.discard_burnin else 0
        row0 = max(offset, de.n_initial)
        out = h.power_posterior(row0, h.n_rows - row0)
        arr = h.chains(offset, max(n_iter // h.store_every - offset, 0))
        top = arr[(K - 1) * de.n_groups * de.Np:]           # the particles of the t = 1 rung
        names = _flat_names(model.names, shapes) + ["acceptance", "lp"]
        out["chains"] = Chains(top.transpose(2, 1, 0), names, [str(n) for n in model.names])
        return out
    finally:
        try:
            binding.join()
        except BaseException:                                # noqa: BLE001
            pass
        h.close()


def _comparison_handle(model: DEModel, d, device=0, devices=None):
    """A handle bound to the model's likelihood alone, for the pointwise entry points: no sampler state, no run (they leave the
    priors out, so every parameter gets a flat one here)."""
    ll = model.loglike
    if not isinstance(ll, GPULoglike):
        raise TypeError("loglike must be a GPULoglike: only a model that runs on the device has pointwise log-likelihoods here")
    n_dev = 1 if devices is None else max(1, len(devices))
    h = Handle(n_dev, 3, d, [-np.inf] * d, [np.inf] * d, device=device, devices=devices)
    try:
        h.set_model(ll.kind, [("flat",)] * d, x=ll.x, choice=ll.choice, sigma=ll.sigma, lba_floor=ll.lba_floor, cov=ll.cov,
                    source=ll.source, n_sim=ll.n_sim, sim_floor=ll.sim_floor)
    except BaseException:
        h.close()
        raise
    return h


def _chain_draws(chains: Chains):
    """The parameter draws of `chains` as theta[n_chains * n_steps][d], chain by chain."""
    v = np.asarray(chains.value)
    d = len(chains.names) - 2
    n_steps, _, n_chains = v.shape
    return np.ascontiguousarray(v[:, :d, :].transpose(2, 0, 1)).reshape(n_chains * n_steps, d), n_steps, n_chains


def pointwise_loglikelihoods(model: DEModel, chains: Chains, device=0, devices=None):
    """log p(y_i | theta) of every observation under every draw of `chains`, computed on the device: an array
    (n_obs, n_steps, n_chains), the [data, step, chain] order ParetoSmooth.psis_loo takes.  Priors are left out; what an
    observation is for each kind is stated at demcmc_eval_pointwise (include/demcmc_b200.h)."""
    theta, n_steps, n_chains = _chain_draws(chains)
    h = _comparison_handle(model, theta.shape[1], device, devices)
    try:
        out = h.eval_pointwise(theta)
    finally:
        h.close()
    return out.reshape(n_chains, n_steps, -1).transpose(2, 1, 0)


def loo(model: DEModel, chains: Chains, device=0, devices=None):
    """PSIS-LOO and WAIC of the model over the draws of `chains` (at most 16384 draws; thin longer chains), Pareto
    smoothing on the device (demcmc_loo, r_eff = 1).  Returns a dict: the totals elpd_loo, se_elpd_loo, p_loo, elpd_waic,
    se_elpd_waic, p_waic and n_bad_k (observations with pareto_k > 0.7), and the per-observation arrays elpd_loo_i,
    pareto_k, lppd_i, p_waic_i."""
    theta, _, _ = _chain_draws(chains)
    h = _comparison_handle(model, theta.shape[1], device, devices)
    try:
        elpd_i, k, lppd_i, pw_i = h.loo(theta)
    finally:
        h.close()
    n = elpd_i.size
    waic_i = lppd_i - pw_i
    elpd = float(elpd_i.sum())
    return {"elpd_loo": elpd, "se_elpd_loo": float(np.sqrt(n * np.var(elpd_i))), "p_loo": float(lppd_i.sum() - elpd),
            "elpd_waic": float(waic_i.sum()), "se_elpd_waic": float(np.sqrt(n * np.var(waic_i))), "p_waic": float(pw_i.sum()),
            "n_bad_k": int(np.sum(k > 0.7)), "elpd_loo_i": elpd_i, "pareto_k": k, "lppd_i": lppd_i, "p_waic_i": pw_i}


class Particle:
    """What optimize returns per particle (src/structs.jl:202-223): Θ (one entry per named parameter),
    weight and id."""

    def __init__(self, Θ, weight, id):
        self.Θ, self.weight, self.id = Θ, weight, id


def optimize(model: DEModel, de: DE, *args, progress=False, device=0, **kwargs):
    """optimize(model, de, n_iter) / optimize(model, de, MCMCThreads(), n_iter) (src/optimize.jl:17-66):
    the same population step with de.update_particle = maximize / minimize and
    de.evaluate_fitness = evaluate_fun; returns vcat(groups...) as a list of Particles."""
    if len(args) == 2 and isinstance(args[0], MCMCThreads):
        n_iter = int(args[1])
    elif len(args) == 1:
        n_iter = int(args[0])
    else:
        raise TypeError("optimize(model, de, n_iter) or optimize(model, de, MCMCThreads(), n_iter)")
    # optimize returns the final particles only (src/optimize.jl:38): no history row is needed, so none but the last is kept
    h, shapes, d, binding = build_handle(model, de, device=device, n_iter=n_iter, store_every=max(1, n_iter), background_model=True)
    try:
        P = de.n_groups * de.Np
        theta0 = _draw_states(model.sample_prior, P, d)
        binding.join()
        h.set_state(theta0)
        h.run(n_iter)
        de.iter = n_iter
        th, w, ids = h.get_state()
    finally:
        try:
            binding.join()
        except BaseException:                                # noqa: BLE001
            pass
        h.close()
    out = []
    for c in range(P):
        Θ, k = [], 0
        for sh in shapes:
            n = int(np.prod(sh)) if len(sh) else 1
            Θ.append(th[c, k:k + n].reshape(sh, order="F") if len(sh) else float(th[c, k]))
            k += n
        out.append(Particle(Θ, float(w[c]), int(ids[c]) + 1))
    return out


def get_optimal(de: DE, model: DEModel, particles):
    """get_optimal (src/utilities.jl:258-266): the best particle's Θ by name and its weight."""
    better = (lambda a, b: a > b) if de.update_particle is maximize else (lambda a, b: a < b)
    mx = particles[0]
    for p in particles:
        if better(p.weight, mx.weight):
            mx = p
    return {str(n): v for n, v in zip(model.names, mx.Θ)}, mx.weight


def bundle_samples(model, de, samples, accept, lp, final_ids, shapes, n_iter):
    """bundle_samples (src/main.jl:222-250), including its quirk: chain c takes its draws from
    samples[:, :, c] (particle id c) but "acceptance"/"lp" from the particle sitting at final
    position c."""
    P, d, _ = samples.shape
    Ns = n_iter - de.burnin if de.discard_burnin else n_iter
    offset = de.burnin if de.discard_burnin else 0
    names = _flat_names(model.names, shapes) + ["acceptance", "lp"]
    v = np.zeros((max(Ns, 0), d + 2, P))
    if Ns > 0:
        v[:, :d, :] = samples[:, :, offset:offset + Ns].transpose(2, 1, 0)
        v[:, d, :] = accept[final_ids, offset:offset + Ns].T
        v[:, d + 1, :] = lp[final_ids, offset:offset + Ns].T
    return Chains(v, names, [str(n) for n in model.names])

"""Power posteriors: tempered groups (demcmc_set_temperatures), the stored untempered log-likelihoods (demcmc_get_loglike) and
the thermodynamic-integration / stepping-stone evidence (demcmc_power_posterior: k_power_posterior, then the split-R-hat and
ESS of demcmc_get_diagnostics on the log-likelihood series).

On the host test double and, with -m gpu, on a B200:
  - every temperature 1 gives the chains, lp and accept of an untempered handle bit for bit;
  - with per-group temperatures, every traced proposal's weight is prior + t loglike of the oracle's own density functions
    (oracle/demcmc_oracle.c), every accept decision is the oracle's accept of those weights, and every stored
    log-likelihood is the oracle's log-likelihood of the stored draw (teacher-forced: each sweep is checked from the
    library's own state before it);
  - the outputs of demcmc_power_posterior match a np.longdouble restatement from the demcmc_get_loglike rows, with the R-hat /
    ESS reference of test_history_summaries.py, and the totals follow the header's formulas;
  - two devices give the bits of one;
  - every refusal.
On a B200 only: the estimates against closed forms (Binomial with a Beta prior) and quadrature (Gaussian (mu, sigma))."""
import math
import os
import subprocess

import numpy as np
import pytest

import common
from common import D, O, make_case
from test_history_summaries import ref_diagnostics

LD = np.longdouble
EINVAL, ESTATE, EUNSUPPORTED = -1, -5, -6

# Tolerances against the longdouble restatement: R-hat and ESS those of test_history_summaries.py (absolute / relative);
# means, log ratios and totals relative to max(|value|, 1), variances relative: float64 sums of at most ~1e5 terms.
TOL_MEAN, TOL_VAR, TOL_ESS, TOL_RHAT = 1e-12, 1e-10, 4e-10, 2e-11


# The plain test double (tests/emu/Makefile) has no power-posterior launchers; tests/emu/emu_power_posterior.cpp holds their
# host versions, built here with the same sources and flags into a test double of its own.
CSRC = os.path.join(common.ROOT, "differentialevolutionmcmc.jl_b200", "csrc")


@pytest.fixture(scope="session")
def pp_emu_lib(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("emu_pp") / "libdemcmc_emu_pp.so")
    emu = os.path.join(common.ROOT, "tests", "emu")
    subprocess.run(["/usr/bin/g++", "-O2", "-fPIC", "-std=c++17", "-ffp-contract=off", "-Wall", "-Wno-unknown-pragmas", "-I", CSRC,
                    "-shared", "-o", out, os.path.join(emu, "emu_backend.cpp"), os.path.join(emu, "emu_power_posterior.cpp"),
                    os.path.join(CSRC, "engine.cpp"), os.path.join(CSRC, "planner.cpp")], check=True)
    return out


@pytest.fixture(params=["emu", pytest.param("cuda", marks=pytest.mark.gpu)])
def backend(request):
    request.getfixturevalue(request.param)
    if request.param == "cuda":
        common.use_cuda()
    else:
        D._ffi.use_library(request.getfixturevalue("pp_emu_lib"))
    return request.param


def test_the_plain_test_double_refuses(emu):
    case = make_case("gaussian", np.random.default_rng(5))
    with case.handle(4, 4, alpha=0.0) as h:
        with pytest.raises(D._ffi.DemcmcError) as e:
            h.set_temperatures([0.0, 0.3, 0.6, 1.0])
        assert e.value.code == EUNSUPPORTED and "no power-posterior kernels" in str(e.value)


def _err(msg_code):
    return pytest.raises(D._ffi.DemcmcError, match=msg_code)


def _run(case, G, Np, n_iter, temps=None, seed=7, rng_seed=1, devices=None, tape=None, **kw):
    """one handle (tempered when temps is given): samples, lp, accept, loglike rows, state, trace"""
    rng = np.random.default_rng(rng_seed)
    theta0 = case.theta0(rng, G * Np)
    kw.setdefault("alpha", 0.0)
    with case.handle(G, Np, seed=seed, trace=True, devices=devices, **kw) as h:
        if temps is not None:
            h.set_temperatures(temps)
        h.set_state(theta0)
        w0 = h.get_state()[1]
        if tape is None:
            h.run(n_iter)
        else:
            h.replay(tape, n_iter)
        out = dict(samples=h.samples(), lp=h.lp(), accept=h.accept(), state=h.get_state(), w0=w0, theta0=theta0)
        if temps is not None:
            out["loglike"] = h.loglike()
            out["trace"] = h.trace()
    return out


def _same(a, b):
    for k in ("samples", "lp", "accept"):
        assert np.array_equal(a[k], b[k], equal_nan=True), k
    for x, y in zip(a["state"], b["state"]):
        assert np.array_equal(x, y, equal_nan=True)


# ---- t = 1 is the untempered sampler ----------------------------------------------------------------------------------
@pytest.mark.parametrize("blocked", [False, True])
def test_all_ones_is_untempered(backend, blocked):
    if blocked:   # the hierarchical model with its two parameter blocks, thinned
        case = make_case("hier_normal", np.random.default_rng(3), n_subjects=5)
        kw = dict(blocks=common.hier_blocks(5), store_every=3, burnin=10, theta_snooker=0.1)
    else:
        case = make_case("gaussian", np.random.default_rng(3))
        kw = dict(burnin=10, theta_snooker=0.1)
    G, Np = 4, 6
    a = _run(case, G, Np, 30, **kw)
    b = _run(case, G, Np, 30, temps=np.ones(G), **kw)
    _same(a, b)


# ---- per-group temperatures, teacher-forced against the oracle's densities and accept -------------------------------------
def _oracle_w(model, lo, hi, t, theta):
    if not np.all((theta >= lo) & (theta <= hi)):
        return -np.inf, O.loglike(model, theta)
    ll = O.loglike(model, theta)
    return O.prior_loglike(model, theta) + (0.0 if t == 0 else t * ll), ll


def _close(a, b, rtol=1e-12):
    if not np.isfinite(b):
        return a == b
    return abs(a - b) <= rtol * max(abs(b), 1.0)


def check_tempered_replay(name, G=4, Np=6, n_iter=12, temps=(0.0, 0.2, 0.2, 1.0)):
    case = make_case(name, np.random.default_rng(11))
    model = case.oracle_model()
    temps = np.asarray(temps)
    rng = np.random.default_rng(1)
    theta0 = case.theta0(rng, G * Np)
    cfg = case.oracle_config(G, Np, seed=7, alpha=0.0, burnin=5, theta_snooker=0.1)
    ref = O.run(cfg, model, theta0, n_iter)
    r = _run(case, G, Np, n_iter, temps=temps, tape=ref["tape"], burnin=5, theta_snooker=0.1)
    P = G * Np
    t_of = np.repeat(temps, Np)
    w = np.empty(P)
    ll = np.empty(P)
    for p in range(P):
        w[p], ll[p] = _oracle_w(model, case.lo, case.hi, t_of[p], theta0[p])
        assert _close(r["w0"][p], w[p]), ("initial weight", p, r["w0"][p], w[p])
    tr, tape = r["trace"], ref["tape"]
    theta = theta0.copy()
    n_acc = 0
    for s in range(n_iter):
        for p in range(P):
            prop = tr["prop_theta"][s, p]
            wp, llp = _oracle_w(model, case.lo, case.hi, t_of[p], prop)
            assert _close(tr["prop_weight"][s, p], wp), ("proposal weight", s, p, tr["prop_weight"][s, p], wp)
            acc = O.accept(tr["prop_weight"][s, p], w[p], tr["log_adj"][s, p], tape["u_acc"][s, p])
            assert bool(tr["accepted"][s, p]) == acc, ("accept", s, p)
            if acc:
                theta[p], w[p], ll[p] = prop, tr["prop_weight"][s, p], llp
                n_acc += 1
        assert np.array_equal(r["samples"][:, :, s], theta), s
        assert np.allclose(r["lp"][:, s], w, rtol=1e-12, atol=0)
        assert np.allclose(r["loglike"][:, s], ll, rtol=1e-12, atol=0)
    assert 0 < n_acc < n_iter * P


@pytest.mark.parametrize("name", ["gaussian", "lba", "binomial"])
def test_tempered_replay_against_the_oracle(backend, name):
    check_tempered_replay(name)


# ---- demcmc_power_posterior against a longdouble restatement ----------------------------------------------------------
def ref_evidence(ll_rows, temps, Np, row0, n):
    """the header's estimator from the loglike rows [P][n_rows], in longdouble"""
    g_t = np.asarray(temps)
    first = [g for g in range(g_t.size) if g == 0 or g_t[g] != g_t[g - 1]] + [g_t.size]
    K = len(first) - 1
    T = [LD(g_t[first[k]]) for k in range(K)]
    rungs = []
    for k in range(K):
        x = ll_rows[first[k] * Np:first[k + 1] * Np, row0:row0 + n]
        v = np.asarray(x, dtype=LD).reshape(-1)
        mean = v.sum() / v.size
        var = ((v - mean) ** 2).sum() / (v.size - 1)
        rhat, ess, _, _ = ref_diagnostics(x)
        lr = me = ve = LD(math.nan)
        if k + 1 < K:
            dl = T[k + 1] - T[k]
            m = v.max()
            e = np.exp(dl * (v - m))
            me = e.sum() / e.size
            ve = ((e - me) ** 2).sum() / (e.size - 1)
            lr = np.log(me) + dl * m
        rungs.append(dict(mean=mean, var=var, ess=LD(ess), rhat=LD(rhat), lr=lr, me=me, ve=ve))
    ti = sum((T[k + 1] - T[k]) * (rungs[k]["mean"] + rungs[k + 1]["mean"]) / 2 for k in range(K - 1))
    corr = sum((T[k + 1] - T[k]) ** 2 * (rungs[k + 1]["var"] - rungs[k]["var"]) / 12 for k in range(K - 1))
    wts = [((T[k] - T[k - 1] if k > 0 else 0) + (T[k + 1] - T[k] if k + 1 < K else 0)) / 2 for k in range(K)]
    se_ti = np.sqrt(sum(wts[k] ** 2 * rungs[k]["var"] / rungs[k]["ess"] for k in range(K)))
    se_ss = np.sqrt(sum(rungs[k]["ve"] / (rungs[k]["ess"] * rungs[k]["me"] ** 2) for k in range(K - 1)))
    return dict(t=[float(x) for x in T], rungs=rungs, log_z_ti=ti, log_z_ti2=ti - corr, log_z_ss=sum(r["lr"] for r in rungs[:-1]),
                se_ti=se_ti, se_ss=se_ss)


def check_evidence(out, ref):
    assert out["n_rungs"] == len(ref["rungs"])
    assert np.array_equal(out["t"], ref["t"])
    for k, r in enumerate(ref["rungs"]):
        assert abs(out["mean_ll"][k] - float(r["mean"])) <= TOL_MEAN * max(abs(float(r["mean"])), 1.0), k
        assert abs(out["var_ll"][k] - float(r["var"])) <= TOL_VAR * float(r["var"]), k
        assert abs(out["ess_ll"][k] - float(r["ess"])) <= TOL_ESS * float(r["ess"]), k
        assert abs(out["rhat_ll"][k] - float(r["rhat"])) <= TOL_RHAT, k
        if k + 1 < len(ref["rungs"]):
            assert abs(out["log_ratio"][k] - float(r["lr"])) <= TOL_MEAN * max(abs(float(r["lr"])), 1.0), k
        else:
            assert np.isnan(out["log_ratio"][k])
    for key in ("log_z_ti", "log_z_ti2", "log_z_ss"):
        assert abs(out[key] - float(ref[key])) <= TOL_MEAN * max(abs(float(ref[key])), 1.0), key
    for key in ("se_ti", "se_ss"):
        assert abs(out[key] - float(ref[key])) <= TOL_ESS * float(ref[key]), key


TEMPS = np.array([0.0, 0.0, 0.05, 0.05, 0.3, 0.3, 1.0, 1.0])    # four rungs of two groups


def _evidence_run(case, n_iter, devices=None, store_every=1, n_initial=0, row0=None):
    G, Np = TEMPS.size, 4
    rng = np.random.default_rng(2)
    with case.handle(G, Np, seed=9, alpha=0.0, burnin=0, devices=devices, store_every=store_every, n_initial=n_initial) as h:
        h.set_temperatures(TEMPS)
        if n_initial:
            h.set_history(np.stack([case.theta0(rng, G * Np) for _ in range(n_initial)]))
            h.set_state(None)
        else:
            h.set_state(case.theta0(rng, G * Np))
        h.run(n_iter)
        r0 = n_initial if row0 is None else row0
        return h.power_posterior(r0, h.n_rows - r0), h.loglike(), h.n_rows


@pytest.mark.parametrize("n_iter,store_every,n_initial", [(300, 1, 0), (701, 2, 3), (1030, 1, 0)])
def test_evidence_matches_the_restatement(backend, n_iter, store_every, n_initial):
    case = make_case("gaussian", np.random.default_rng(5))
    out, ll, n_rows = _evidence_run(case, n_iter, store_every=store_every, n_initial=n_initial)
    assert np.all(np.isnan(ll[:, :n_initial])) and np.all(np.isfinite(ll[:, n_initial:]))
    check_evidence(out, ref_evidence(ll, TEMPS, 4, n_initial, n_rows - n_initial))


def test_loglike_rows_are_the_oracle_loglike_of_the_draws(backend):
    case = make_case("lnr", np.random.default_rng(5))
    G, Np = 4, 5
    r = _run(case, G, Np, 20, temps=[0.0, 0.4, 0.7, 1.0], burnin=5)
    model = case.oracle_model()
    s, ll = r["samples"], r["loglike"]
    for p in range(G * Np):
        for row in range(s.shape[2]):
            assert _close(ll[p, row], O.loglike(model, s[p, :, row]))


def test_two_devices_give_the_bits_of_one(backend):
    if backend == "cuda" and D._ffi.lib().demcmc_device_count() < 2:
        pytest.skip("one GPU")
    case = make_case("gaussian", np.random.default_rng(5))
    a = _evidence_run(case, 300)
    b = _evidence_run(case, 300, devices=[0, 1])
    assert np.array_equal(a[1], b[1])
    for k in a[0]:
        assert np.array_equal(np.asarray(a[0][k]), np.asarray(b[0][k]), equal_nan=True), k


def test_repeated_calls_give_the_same_bits(backend):
    case = make_case("gaussian", np.random.default_rng(5))
    G, Np = TEMPS.size, 4
    with case.handle(G, Np, seed=9, alpha=0.0, burnin=0) as h:
        h.set_temperatures(TEMPS)
        h.set_state(case.theta0(np.random.default_rng(2), G * Np))
        h.run(200)
        a, b = h.power_posterior(), h.power_posterior()
    for k in a:
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k]), equal_nan=True), k


# ---- refusals ---------------------------------------------------------------------------------------------------------
def test_refusals(backend):
    case = make_case("gaussian", np.random.default_rng(5))
    G, Np = 4, 4
    th = case.theta0(np.random.default_rng(2), G * Np)
    ladder = [0.0, 0.3, 0.6, 1.0]
    with case.handle(G, Np, alpha=0.0) as h:
        for bad in ([0.0, 0.3, np.nan, 1.0], [0.0, 0.3, 1.2, 1.0], [-0.1, 0.3, 0.6, 1.0], [0.0, 1.0]):
            with _err("temperature|groups"):
                h.set_temperatures(bad)
        with _err("no temperatures"):
            h.power_posterior(0, 4)
    h = D.Handle(G, Np, case.d, case.lo, case.hi, alpha=0.0)
    with h:
        with _err("set_model must come before"):
            h.set_temperatures(ladder)
        h.set_model(case.kind, case.prior, **case.data)
        h.set_state(th)
        with _err("before set_state"):
            h.set_temperatures(ladder)
        with _err("not tempered"):
            h.loglike()
    for kw, what in ((dict(alpha=0.1), "alpha = 0"), (dict(alpha=0.0, update="maximize"), "mh_update"),
                     (dict(alpha=0.0, fitness="fun"), "mh_update")):
        with case.handle(G, Np, **kw) as h, _err(what):
            h.set_temperatures(ladder)
    with case.handle(G, Np, alpha=0.0, n_initial=2, resample=True) as h, _err("resample"):
        h.set_temperatures(ladder)
    with case.handle(G, Np, alpha=0.0, burnin=0) as h:
        h.set_temperatures(ladder)
        h.set_state(th)
        with _err("saved weights"):
            h.set_weights(np.zeros(G * Np))
        h.run(10)
        with _err("at least 4 rows"):
            h.power_posterior(0, 3)
        with _err("cap"):
            ev = D._ffi.Evidence()
            D._ffi.check(D._ffi.lib().demcmc_power_posterior(h._h, 0, 10, 3, D._ffi.C.byref(ev), None, None, None, None, None, None))
    with case.handle(G, Np, alpha=0.0, n_initial=2) as h:
        h.set_temperatures(ladder)
        h.set_history(np.stack([th, th]))
        h.set_state(None)
        h.run(10)
        with _err("n_initial"):
            h.power_posterior(1, 8)
    for bad in ([0.3, 0.3, 0.6, 1.0], [0.0, 0.6, 0.3, 1.0], [0.0, 0.3, 0.6, 0.9]):
        with case.handle(G, Np, alpha=0.0) as h:
            h.set_temperatures(bad)
            h.set_state(th)
            h.run(10)
            with _err("increase"):
                h.power_posterior(0, 10)
    flat = [("flat",), ("halfcauchy", 0, 1)]
    with D.Handle(G, Np, 2, case.lo, case.hi, alpha=0.0) as h:
        h.set_model("gaussian", flat, **case.data)
        h.set_temperatures(ladder)
        h.set_state(th)
        h.run(10)
        with _err("improper"):
            h.power_posterior(0, 10)
    # a replay tape that migrates
    cfg = case.oracle_config(G, Np, seed=7, alpha=0.9)
    ref = O.run(cfg, case.oracle_model(), th, 5)
    assert ref["tape"]["mig_n"].max() > 0
    with case.handle(G, Np, alpha=0.0) as h:
        h.set_temperatures(ladder)
        h.set_state(th)
        with _err("migrates"):
            h.replay(ref["tape"], 5)


def test_api_refuses_migration_and_returns_the_top_rung(backend):
    rng = np.random.default_rng(0)
    x = rng.normal(0.5, 1.0, 40)
    model = D.DEModel(loglike=D.GPULoglike("gaussian", x), prior_loglike=D.GPUPrior(D.Normal(0, 10), D.HalfCauchy(0, 1)),
                      names=("mu", "sigma"), sample_prior=lambda: (rng.normal(0, 1), abs(rng.standard_cauchy()) + 0.1))
    de = D.DE(n_groups=2, Np=6, burnin=50, bounds=((-np.inf, np.inf), (0, np.inf)), sample_prior=model.sample_prior, seed=3)
    with pytest.raises(ValueError, match="α = 0"):
        D.power_posterior(model, de, 100, n_temperatures=4)
    de = D.DE(n_groups=2, Np=6, burnin=50, bounds=((-np.inf, np.inf), (0, np.inf)), sample_prior=model.sample_prior, seed=3, α=0.0)
    out = D.power_posterior(model, de, 200, n_temperatures=5, power=4.0)
    assert out["n_rungs"] == 5 and np.allclose(out["t"], (np.arange(5) / 4.0) ** 4)
    assert out["chains"].value.shape == (150, 4, 12)
    assert np.all(np.isfinite([out["log_z_ti"], out["log_z_ti2"], out["log_z_ss"], out["se_ti"], out["se_ss"]]))


# ---- on a B200: every path, t = 1 against untempered ---------------------------------------------------------------------
CUSTOM_GAUSSIAN = r"""
#define DEMCMC_NPAR 2
__device__ void demcmc_prepare(const double *theta, double *par) { par[0] = theta[0]; par[1] = log(theta[1]); }
__device__ double demcmc_obs(const double *par, const double *x)
{ const double z = (x[0] - par[0]) * exp(-par[1]); return -0.5 * z * z - par[1] - 0.91893853320467274178; }
"""


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["persistent", "single_cta", "wide", "level_by_level", "custom"])
def test_all_ones_on_every_path(cuda, monkeypatch, path):
    rng = np.random.default_rng(4)
    kw = dict(burnin=5, theta_snooker=0.1)
    G, Np, n_iter = 4, 6, 20
    if path in ("persistent", "level_by_level"):
        case = make_case("mvnormal", rng, n_obs=3000, n_dim=50)
        Np = 256
        monkeypatch.setenv("DEMCMC_PERSIST", "1" if path == "persistent" else "0")
    elif path == "single_cta":
        case = make_case("gaussian", rng)
    elif path == "wide":
        case = make_case("hier_normal", rng, n_subjects=300, n_obs=8)
        Np, n_iter = 32, 10
        kw["blocks"] = common.hier_blocks(300)
        monkeypatch.setenv("DEMCMC_PERSIST", "0")
    else:
        case = make_case("gaussian", rng)
        case.kind = "custom"
        case.data = dict(x=case.data["x"], source=CUSTOM_GAUSSIAN)
    a = _run(case, G, Np, n_iter, **kw)
    b = _run(case, G, Np, n_iter, temps=np.ones(G), **kw)
    _same(a, b)


# ---- on a B200: the estimates against exact answers --------------------------------------------------------------------
def _ladder(K, power=4.0):
    return (np.arange(K) / (K - 1)) ** power


@pytest.mark.gpu
def test_binomial_beta_closed_form(cuda):
    from scipy.special import betaln, digamma, gammaln
    a, b, N, k = 2.0, 3.0, 40, 13
    K, Gk, Np, n_iter, burn = 16, 2, 16, 6000, 1000
    T = _ladder(K)
    temps = np.repeat(T, Gk)
    with D.Handle(K * Gk, Np, 1, [0.0], [1.0], alpha=0.0, burnin=0, seed=31) as h:
        h.set_model("binomial", [("beta", a, b)], x=np.array([float(N), float(k)]))
        h.set_temperatures(temps)
        h.set_state(np.random.default_rng(1).beta(a, b, (K * Gk * Np, 1)))
        h.run(n_iter)
        out = h.power_posterior(burn, h.n_rows - burn)
    lc = gammaln(N + 1) - gammaln(k + 1) - gammaln(N - k + 1)
    # E_t[log L] under the power posterior Beta(a + t k, b + t (N - k))
    A, B = a + T * k, b + T * (N - k)
    exact_mean = lc + k * (digamma(A) - digamma(A + B)) + (N - k) * (digamma(B) - digamma(A + B))
    mcse = np.sqrt(out["var_ll"] / out["ess_ll"])
    assert np.all(np.abs(out["mean_ll"] - exact_mean) <= 4 * mcse + 1e-12), (out["mean_ll"] - exact_mean) / mcse
    dl = np.diff(T)
    trap_exact = np.sum(dl * (exact_mean[:-1] + exact_mean[1:]) / 2)
    assert abs(out["log_z_ti"] - trap_exact) <= 4 * out["se_ti"]
    log_z = lc + betaln(a + k, b + N - k) - betaln(a, b)
    # ladder bias of the corrected trapezoid and of the stepping stones at 16 rungs with power 4: stated bound 0.02 nats
    assert abs(out["log_z_ti2"] - log_z) <= 4 * out["se_ti"] + 0.02, (out["log_z_ti2"], log_z)
    assert abs(out["log_z_ss"] - log_z) <= 4 * out["se_ss"] + 0.02, (out["log_z_ss"], log_z)
    assert np.all(out["rhat_ll"] < 1.05)


@pytest.mark.gpu
def test_gaussian_against_quadrature(cuda):
    from scipy import integrate, stats
    rng = np.random.default_rng(17)
    x = rng.normal(0.7, 1.3, 50)
    n, xbar, ss = x.size, x.mean(), ((x - x.mean()) ** 2).sum()
    K, Gk, Np, n_iter, burn = 24, 2, 12, 6000, 1000
    T = _ladder(K)
    prior = [("normal", 0, 10), ("halfcauchy", 0, 1)]      # gaussian_tests.jl: mu ~ Normal(0, 10), sigma ~ HalfCauchy(0, 1)
    lo, hi = [-np.inf, 0.0], [np.inf, np.inf]
    P = K * Gk * Np
    th0 = np.column_stack([rng.normal(0, 10, P), np.abs(rng.standard_cauchy(P))])
    with D.Handle(K * Gk, Np, 2, lo, hi, alpha=0.0, burnin=0, seed=5, theta_snooker=0.1) as h:
        h.set_model("gaussian", prior, x=x)
        h.set_temperatures(np.repeat(T, Gk))
        h.set_state(th0)
        h.run(n_iter)
        out = h.power_posterior(burn, h.n_rows - burn)
        s = h.samples()[:, :, burn:]

    # p(y | sigma) with mu integrated analytically: N(y; mu 1, sigma^2 I) N(mu; 0, 100)
    def log_like_sigma(sig):
        v = sig * sig
        prec = n / v + 1.0 / 100.0
        return (-0.5 * n * math.log(2 * math.pi * v) - 0.5 * ss / v - 0.5 * math.log(100.0 * prec)
                - 0.5 * (n * xbar * xbar / v) + 0.5 * (n * xbar / v) ** 2 / prec)
    pr_sig = lambda sg: 2.0 / (math.pi * (1 + sg * sg))     # noqa: E731
    peak = max(log_like_sigma(sg) for sg in np.linspace(0.3, 5, 400))
    Z = integrate.quad(lambda sg: pr_sig(sg) * math.exp(log_like_sigma(sg) - peak), 0, np.inf, limit=200)[0]
    log_z = peak + math.log(Z)
    # stepping stones only: under the HalfCauchy prior the t = 0 rung reaches sigma near 0, where the log-likelihood is of
    # order -1e10 (var_ll[0] ~ 1e21 on the test double), and the trapezoid rules over the rung means do not converge
    assert abs(out["log_z_ss"] - log_z) <= 4 * out["se_ss"] + 0.02, (out["log_z_ss"], log_z)
    # the t = 1 rung's posterior moments (sigma's marginal by quadrature, mu's from its conditional normal)
    top = s[(K - 1) * Gk * Np:]
    w = lambda sg: pr_sig(sg) * math.exp(log_like_sigma(sg) - peak) / Z     # noqa: E731
    m_sig = integrate.quad(lambda sg: sg * w(sg), 0, np.inf)[0]
    sd_sig = math.sqrt(integrate.quad(lambda sg: (sg - m_sig) ** 2 * w(sg), 0, np.inf)[0])
    cond = lambda sg: ((n * xbar / sg ** 2) / (n / sg ** 2 + 0.01), 1.0 / (n / sg ** 2 + 0.01))   # noqa: E731
    m_mu = integrate.quad(lambda sg: cond(sg)[0] * w(sg), 0, np.inf)[0]
    sd_mu = math.sqrt(integrate.quad(lambda sg: (cond(sg)[1] + cond(sg)[0] ** 2) * w(sg), 0, np.inf)[0] - m_mu ** 2)
    assert abs(top[:, 0, :].mean() - m_mu) < 0.1 * sd_mu and abs(top[:, 0, :].std() / sd_mu - 1) < 0.1
    assert abs(top[:, 1, :].mean() - m_sig) < 0.1 * sd_sig and abs(top[:, 1, :].std() / sd_sig - 1) < 0.1
    # the t = 0 rung samples the prior: mu ~ Normal(0, 10), sigma ~ HalfCauchy(0, 1) (median 1)
    bot = s[:Gk * Np]
    assert abs(bot[:, 0, :].mean()) < 1.5 and abs(bot[:, 0, :].std() / 10 - 1) < 0.1
    assert abs(np.median(bot[:, 1, :]) / stats.halfcauchy.median() - 1) < 0.1

"""Model comparison on the device: pointwise log-likelihoods (demcmc_eval_pointwise) and PSIS-LOO / WAIC (demcmc_loo).

The reference is in this file: `ref_psis` restates the estimator of include/demcmc_b200.h (demcmc_loo) step by step in
numpy, with every sum, exponential and logarithm in np.longdouble; the log ratios x_s = min(ll) - ll_s are formed in
float64, as the contract defines them, so the tail holds the same draws.  The reference is checked on its own first: its
GPD fit recovers known shapes from scipy.stats.genpareto samples, and on a conjugate normal model its elpd_loo matches the
exact leave-one-out predictive.

CPU (host-only test double): the pointwise values of every registered kind against scipy / the oracle's per-trial forms,
their sum against demcmc_eval, loo against the reference for S in {2, 7, 20, 21, 100, 4000, 16384} (tail cutoffs 4 / 5,
the cap, ties, constant columns), the NaN rule, the refusals, the observation chunks and the slices of a multi-device handle; these
run on a test double built here with the host launchers of tests/emu/emu_loo.cpp (the plain one refuses both calls).  GPU (-m gpu): the same at 1e5
observations, custom sources against the registered kernels, loo at the configs[2] shape and at the cap, the conjugate
model end to end through sample(), an outlier, and bitwise determinism on one and two devices.

Tolerances are 100x the worst error measured on the test double and on one B200 (1000 W power limit), over the inputs
of these tests:
  pointwise, relative to max(1, |value|):  test double 1.5e-15;  B200 1.5e-14 (LBA: the device's exp / erfcx forms)
  sum of the pointwise values vs demcmc_eval, relative to max(1, |ll|):  test double 9.4e-16;  B200 1.8e-16
  loo outputs vs the reference, absolute:  test double 5.8e-13;  B200 3.3e-13 (elpd_loo at S = 16384; pareto_k 4.4e-14)
An infinite k-hat must match exactly.
"""
import math
import os
import subprocess

import numpy as np
import pytest
import scipy.stats as st

import common
from common import D, O, lba_sim, lnr_sim

TOL_PW = 1.5e-12          # pointwise densities
TOL_SUM = 9.4e-14         # their sum against demcmc_eval
TOL_LOO = 5.8e-11         # loo outputs against ref_psis
LD = np.longdouble
DBL_MIN = np.finfo(np.float64).tiny
EPS = np.finfo(np.float64).eps


# ---- the reference ---------------------------------------------------------------------------------------------------
def ref_lse(a):
    m = a.max()
    return m + np.log(np.sum(np.exp(a - m)))


def ref_gpdfit(y):
    """Zhang & Stephens (2009) on the sorted tail y (ArviZ _gpdfit): (k-hat with the prior adjustment, sigma)."""
    y = np.asarray(y, dtype=LD)
    n = y.size
    m = 30 + int(math.sqrt(n))
    b = 1 - np.sqrt(LD(m) / (np.arange(1, m + 1, dtype=LD) - LD(0.5)))
    b /= 3 * y[int(n / 4 + 0.5) - 1]
    b += 1 / y[-1]
    kbar = np.log1p(-b[:, None] * y).mean(axis=1)
    prof = n * (np.log(-(b / kbar)) - kbar - 1)
    w = 1 / np.exp(prof[None, :] - prof[:, None]).sum(axis=1)
    keep = w >= 10 * EPS
    w, b = w[keep], b[keep]
    w = w / w.sum()
    bp = np.sum(b * w)
    k = np.log1p(-bp * y).mean()
    sigma = -k / bp
    return (n * k + 5) / (n + 10), sigma


def ref_gpinv(p, k, sigma):
    if not sigma > 0:
        return np.full(p.shape, np.nan, dtype=LD)
    x = -np.log1p(-p) if abs(k) < EPS else np.expm1(-k * np.log1p(-p)) / k
    return x * sigma


def ref_psis(ll):
    """(elpd_loo, pareto_k, lppd, p_waic) of one observation's S log-likelihoods, as demcmc_loo defines them."""
    ll = np.asarray(ll, dtype=np.float64)
    S = ll.size
    if not np.all(np.isfinite(ll)):
        return (np.nan,) * 4
    L = ll.astype(LD)
    lppd = ref_lse(L) - np.log(LD(S))
    p_waic = np.sum((L - L.sum() / S) ** 2) / (S - 1)
    x64 = ll.min() - ll                                                  # 1. the shifted log ratios
    M = int(math.ceil(min(0.2 * S, 3 * math.sqrt(S))))                   # 2.
    cutoff = max(np.sort(x64)[S - 1 - M], math.log(DBL_MIN))
    tail = np.flatnonzero(x64 > cutoff)
    tail = tail[np.argsort(x64[tail], kind="stable")]                    # (value, draw) order
    x = x64.astype(LD)
    k = np.inf                                                           # 3.
    if tail.size > 4:                                                    # 4.
        ec = np.exp(LD(cutoff))
        k, sigma = ref_gpdfit(np.exp(x[tail]) - ec)
        if np.isfinite(k):                                               # 5.
            sm = np.log(ref_gpinv((np.arange(tail.size, dtype=LD) + LD(0.5)) / tail.size, k, sigma) + ec)
            x[tail] = sm
            x[x > 0] = 0
    lw = x - ref_lse(x)                                                  # 6.
    return float(ref_lse(lw + L)), float(k), float(lppd), float(p_waic)  # 7.


def ref_loo(ll_obs_major):
    return np.array([ref_psis(r) for r in ll_obs_major]).T


def abs_err(a, b):
    """max |a - b|; non-finite entries must agree exactly"""
    a, b = np.asarray(a, float), np.asarray(b, float)
    fin = np.isfinite(b)
    if not (np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(a[np.isinf(b)], b[np.isinf(b)])):
        return np.inf
    return float(np.max(np.abs(a[fin] - b[fin]))) if fin.any() else 0.0


# ---- the reference on its own ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("k_true", [0.2, 0.5, 0.9])
def test_reference_gpdfit_recovers_the_shape(k_true):
    # 4000 GPD(k, 1) samples: the fit's standard error is about (1 + k) / sqrt(n) = 0.019 .. 0.030; allow 4 of them
    n = 4000
    y = np.sort(st.genpareto.rvs(k_true, scale=1.0, size=n, random_state=np.random.default_rng(int(k_true * 100))))
    k, sigma = ref_gpdfit(y)
    assert abs(float(k) - k_true) < 4 * (1 + k_true) / math.sqrt(n), (k, k_true)
    assert abs(float(sigma) - 1.0) < 0.1, sigma


def conjugate(seed=4, n=50, tau=2.0, S=4000):
    """y_i ~ N(mu, 1), mu ~ N(0, tau^2): exact posterior draws, and the exact elpd_loo"""
    rng = np.random.default_rng(seed)
    y = rng.normal(0.7, 1.0, n)
    prec = 1 / tau ** 2 + n
    mu = rng.normal(y.sum() / prec, 1 / math.sqrt(prec), S)
    prec_i = prec - 1
    exact = st.norm.logpdf(y, (y.sum() - y) / prec_i, np.sqrt(1 + 1 / prec_i)).sum()
    return y, mu, exact, tau


def test_reference_matches_exact_loo_on_a_conjugate_model():
    y, mu, exact, _ = conjugate()
    ll = st.norm.logpdf(y[:, None], mu[None, :], 1.0)                   # [obs][draw]
    elpd = ref_loo(ll)[0]
    # p(y_i | y_-i) = 1 / E[1 / p(y_i | mu)]: the Monte-Carlo standard error of its log is sd(1/p) / (mean(1/p) sqrt(S));
    # summed over the observations it bounds the error of the total.  Allow 4 of them.
    inv = np.exp(-ll)
    mc = float(np.sum(inv.std(axis=1) / inv.mean(axis=1)) / math.sqrt(mu.size))
    assert abs(elpd.sum() - exact) < 4 * mc, (elpd.sum(), exact, mc)


# ---- models ----------------------------------------------------------------------------------------------------------
def lnr_logpdf(th, rt, choice):
    """LNR, sigma = 1: winner LogNormal logpdf + losers LogNormal logccdf of rt - tau (vectorised over trials)"""
    t = rt - th[-1]
    with np.errstate(all="ignore"):
        lx = np.log(t)
        z = lx[:, None] - np.asarray(th[:-1])[None, :]
        win = np.arange(z.shape[1])[None, :] == (choice - 1)[:, None]
        v = np.where(win, st.norm.logpdf(z) - lx[:, None], st.norm.logsf(z)).sum(axis=1)
    return np.where(t > 0, v, -np.inf)


def lba_logpdf(th, rt, choice, floor=1e-10):
    """LBA, sd 1 (Brown & Heathcote 2008) with the density floor (vectorised over trials)"""
    na = th.size - 3
    nu, A, k, tau = th[:na], th[na], th[na + 1], th[na + 2]
    b = A + k
    dt = rt - tau
    with np.errstate(all="ignore"):
        den = np.ones_like(rt)
        for r in range(na):
            v = nu[r]
            n1, n2 = (b - A - dt * v) / dt, (b - dt * v) / dt
            c1, c2, p1, p2 = st.norm.cdf(n1), st.norm.cdf(n2), st.norm.pdf(n1), st.norm.pdf(n2)
            f = np.maximum((-v * c1 + p1 + v * c2 - p2) / A, 0.0)
            F = np.maximum(1 + ((b - A - dt * v) / A) * c1 - ((b - dt * v) / A) * c2 + (dt / A) * p1 - (dt / A) * p2, 0.0)
            den *= np.where(choice - 1 == r, f, 1 - F)
        den /= 1 - np.prod(st.norm.cdf(-nu))
        out = np.log(np.maximum(den, floor))
    return np.where(rt < tau, math.log(floor), out)


def model_case(kind, rng, n):
    """(handle kwargs of set_model, d, draws(S), scipy pointwise(theta) -> [n_obs])"""
    if kind == "gaussian":
        x = rng.normal(0.3, 1.2, n)
        return dict(x=x), 2, lambda S: np.column_stack([rng.normal(0.3, 0.1, S), rng.uniform(1.0, 1.4, S)]), \
            lambda th: st.norm.logpdf(x, th[0], th[1])
    if kind == "mvnormal":
        dm = 7
        mu = rng.normal(size=dm)
        x = rng.normal(mu, 1.1, size=(n, dm))
        return dict(x=x), dm + 1, lambda S: np.column_stack([rng.normal(mu, 0.05, (S, dm)), rng.uniform(1.0, 1.2, S)]), \
            lambda th: st.multivariate_normal.logpdf(x, th[:dm], th[dm] ** 2 * np.eye(dm))
    if kind == "mvnormal_full":
        dm = 6
        A = rng.normal(size=(dm, dm))
        cov = A @ A.T + 0.5 * np.eye(dm)
        mu = rng.normal(size=dm)
        x = rng.multivariate_normal(mu, 1.3 ** 2 * cov, size=n)
        return dict(x=x, cov=cov), dm + 1, lambda S: np.column_stack([rng.normal(mu, 0.1, (S, dm)), rng.uniform(1.2, 1.4, S)]), \
            lambda th: st.multivariate_normal.logpdf(x, th[:dm], th[dm] ** 2 * cov)
    if kind == "hier_normal":
        subj = 9
        per = max(1, n // subj)
        b0 = rng.normal(0, 1, subj)
        y = rng.normal(1.0 + b0[:, None], 0.5, size=(subj, per))
        return dict(x=y), subj + 3, \
            lambda S: np.column_stack([rng.normal(1, 0.1, S), rng.uniform(0.8, 1.2, S), rng.normal(b0, 0.1, (S, subj)), rng.uniform(0.4, 0.6, S)]), \
            lambda th: st.norm.logpdf(y, th[0] + th[2:2 + subj, None], th[subj + 2]).reshape(-1)
    if kind == "binomial":
        return dict(x=np.array([10.0, 4.0])), 1, lambda S: rng.uniform(0.2, 0.6, (S, 1)), lambda th: np.array([st.binom.logpmf(4, 10, th[0])])
    if kind == "lnr":
        choice, rt = lnr_sim(rng, n)
        return dict(x=rt, choice=choice, n_dim=4), 5, \
            lambda S: np.column_stack([rng.normal([-2, -2, -3, -3], 0.1, (S, 4)), rng.uniform(0.3, 0.45, S)]), \
            lambda th: lnr_logpdf(th, rt, choice)
    if kind == "lba":
        choice, rt = lba_sim(rng, n) if n <= 2000 else lba_vec(rng, n)
        return dict(x=rt, choice=choice, n_dim=2), 5, \
            lambda S: np.column_stack([rng.normal([3, 2], 0.1, (S, 2)), rng.normal(0.8, 0.02, S), rng.normal(0.2, 0.02, S), rng.uniform(0.25, 0.3, S)]), \
            lambda th: lba_logpdf(th, rt, choice)
    raise KeyError(kind)


def lba_vec(rng, n):
    import sys
    sys.path.insert(0, common.os.path.join(common.ROOT, "scripts"))
    from bench_configs import lba_sim_vec
    return lba_sim_vec(rng, n)


def bound(kind, kw, d, devices=None):
    h = D.Handle(1 if devices is None else len(devices), 3, d, [-np.inf] * d, [np.inf] * d, devices=devices)
    h.set_model(kind, [("flat",)] * d, **kw)
    return h


KINDS = ["gaussian", "mvnormal", "mvnormal_full", "hier_normal", "binomial", "lnr", "lba"]


def check_pointwise(kind, n, S, seed=11):
    rng = np.random.default_rng(seed)
    kw, d, draws, ref = model_case(kind, rng, n)
    th = draws(S)
    with bound(kind, kw, d) as h:
        pw = h.eval_pointwise(th)
        ll, _ = h.eval(th)
        part = h.eval_pointwise(th, obs0=h.n_obs // 3, n_obs=h.n_obs // 3)
    want = np.array([ref(t) for t in th])
    assert pw.shape == want.shape
    err = common.rel_err(pw, want)
    assert err < TOL_PW, (kind, err)
    assert np.array_equal(part, pw[:, pw.shape[1] // 3: pw.shape[1] // 3 + pw.shape[1] // 3])
    tot = pw.astype(LD).sum(axis=1)
    serr = float(np.max(np.abs(tot - ll) / np.maximum(1.0, np.abs(ll))))
    assert serr < TOL_SUM, (kind, serr)
    return pw


# ---- CPU: the host-only test double ----------------------------------------------------------------------------------
# The plain test double (tests/emu/Makefile) has no model-comparison launchers; tests/emu/emu_loo.cpp holds their host
# versions, built here with the same sources and flags into a test double of its own.
CSRC = os.path.join(common.ROOT, "differentialevolutionmcmc.jl_b200", "csrc")


@pytest.fixture(scope="session")
def loo_emu_lib(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("emu_loo") / "libdemcmc_emu_loo.so")
    emu = os.path.join(common.ROOT, "tests", "emu")
    subprocess.run(["/usr/bin/g++", "-O2", "-fPIC", "-std=c++17", "-ffp-contract=off", "-Wall", "-Wno-unknown-pragmas", "-I", CSRC,
                    "-shared", "-o", out, os.path.join(emu, "emu_backend.cpp"), os.path.join(emu, "emu_loo.cpp"),
                    os.path.join(CSRC, "engine.cpp"), os.path.join(CSRC, "planner.cpp")], check=True)
    return out


@pytest.fixture
def loo_emu(loo_emu_lib):
    D._ffi.use_library(loo_emu_lib)
    yield


def test_the_plain_test_double_refuses(emu):
    with bound("gaussian", dict(x=np.zeros(5)), 2) as h:
        for call in (lambda: h.loo(np.ones((4, 2))), lambda: h.eval_pointwise(np.ones((4, 2)))):
            with pytest.raises(D._ffi.DemcmcError) as e:
                call()
            assert e.value.code == -6 and "no pointwise kernels" in str(e.value)


@pytest.mark.parametrize("kind", KINDS)
def test_pointwise_matches_scipy(loo_emu, kind):
    check_pointwise(kind, 200, 6)


@pytest.mark.parametrize("kind", ["lnr", "lba"])
def test_pointwise_matches_the_oracle_per_trial(loo_emu, kind):
    rng = np.random.default_rng(5)
    kw, d, draws, ref = model_case(kind, rng, 60)
    th = draws(4)
    with bound(kind, kw, d) as h:
        pw = h.eval_pointwise(th)
    want = np.zeros_like(pw)
    for i in range(60):
        one = O.Model(kind, d, [("flat",)] * d, x=kw["x"][i:i + 1], choice=kw["choice"][i:i + 1], n_dim=kw["n_dim"])
        for s in range(4):
            want[s, i] = O.loglike(one, th[s])
    assert common.rel_err(pw, want) < TOL_PW
    # ... and the vectorised forms the GPU tests use agree with the oracle's
    assert common.rel_err(np.array([ref(t) for t in th]), pw) < 1e-12


def gauss_loo_inputs(S, n=12, seed=3, ties=False, constant=False):
    rng = np.random.default_rng(seed)
    x = np.concatenate([rng.normal(0, 1, n - 1), [4.5]])              # one observation far in the tail
    th = np.column_stack([rng.normal(0.0, 0.3, S), np.abs(rng.normal(1.0, 0.15, S)) + 0.05])
    if ties:
        th[S // 2:] = th[: S - S // 2]                                   # every draw twice (S odd: one three times)
    if constant:
        th[:] = th[0]
    return x, th


@pytest.mark.parametrize("S", [2, 7, 20, 21, 100, 4000, 16384])
@pytest.mark.parametrize("variant", ["plain", "ties", "constant"])
def test_loo_matches_the_reference(loo_emu, S, variant):
    x, th = gauss_loo_inputs(S, n=3 if S == 16384 else 12, ties=variant == "ties", constant=variant == "constant")
    with bound("gaussian", dict(x=x), 2) as h:
        got = np.array(h.loo(th))
        ll = h.eval_pointwise(th)
    want = ref_loo(ll.T)
    for q in range(4):
        assert abs_err(got[q], want[q]) < TOL_LOO, (S, variant, q, got[q], want[q])
    if variant == "constant" or S <= 20:
        assert np.all(np.isinf(got[1]))                                  # the tail holds 4 or fewer draws
    if S == 21 and variant == "plain":
        assert np.all(np.isfinite(got[1]))                               # M = 5: smoothed


def test_non_finite_values_give_nan(loo_emu):
    # lba_floor = 0: a trial faster than a draw's tau has density 0 (log -Inf) under that draw only
    rng = np.random.default_rng(8)
    choice, rt = lba_sim(rng, 40)
    th = np.column_stack([rng.normal([3, 2], 0.1, (30, 2)), np.full(30, 0.8), np.full(30, 0.2), np.full(30, 0.25)])
    th[7, 4] = np.sort(rt)[5] + 1e-9                                     # draw 7: tau above the 6 fastest trials
    with bound("lba", dict(x=rt, choice=choice, n_dim=2, lba_floor=0.0), 5) as h:
        got = np.array(h.loo(th))
        ll = h.eval_pointwise(th)
    bad = ~np.all(np.isfinite(ll), axis=0)
    assert bad[np.argsort(rt)[:6]].all() and not bad.all()
    assert np.all(np.isnan(got[:, bad]))
    want = ref_loo(ll.T[~bad])
    for q in range(4):
        assert abs_err(got[q][~bad], want[q]) < TOL_LOO


def test_refusals(loo_emu):
    x, th = gauss_loo_inputs(10)
    h = D.Handle(1, 3, 2, [-np.inf] * 2, [np.inf] * 2)
    with h:
        for call in (lambda: h.loo(th), lambda: h.eval_pointwise(th, n_obs=3)):
            with pytest.raises(D._ffi.DemcmcError) as e:
                call()
            assert e.value.code == -5                                    # DEMCMC_ESTATE: no model yet
        h.set_model("gaussian", [("flat",)] * 2, x=x)
        for bad in (th[:1], np.zeros((0, 2))):
            with pytest.raises(D._ffi.DemcmcError) as e:
                h.loo(bad)
            assert e.value.code == -1                                    # n < 2
        with pytest.raises(D._ffi.DemcmcError) as e:
            h.loo(np.tile(th[:1], (16385, 1)))
        assert e.value.code == -6 and "thin" in str(e.value)             # above DEMCMC_LOO_MAX_DRAWS
        for obs0, n_obs in ((-1, 2), (11, 2), (0, 13), (5, -1)):
            with pytest.raises(D._ffi.DemcmcError) as e:
                h.eval_pointwise(th, obs0=obs0, n_obs=n_obs)
            assert e.value.code == -1, (obs0, n_obs)
        assert h.eval_pointwise(th, obs0=12, n_obs=0).shape == (10, 0)
        assert h.loo(np.tile(th[:1], (16384, 1)))[1].shape == (12,)      # the cap itself is accepted
    with D.Handle(1, 3, 2, [-5.0] * 2, [5.0] * 2, update="minimize", fitness="fun", theta_snooker=0.0) as h:
        h.set_model("rastrigin", [("flat",)] * 2)
        with pytest.raises(D._ffi.DemcmcError) as e:
            h.loo(th)
        assert e.value.code == -1 and "no observations" in str(e.value)


@pytest.mark.parametrize("n_obs", [2047, 2048, 2049])
def test_observation_chunks(loo_emu, n_obs):
    # 2^25 values of scratch: 2048 observations per chunk at S = 16384
    rng = np.random.default_rng(n_obs)
    x = rng.normal(0, 1, n_obs)
    th = np.column_stack([rng.normal(0, 0.05, 16384), rng.uniform(0.9, 1.1, 16384)])
    with bound("gaussian", dict(x=x), 2) as h:
        got = np.array(h.loo(th))
        pw = h.eval_pointwise(th)
    want_pw = st.norm.logpdf(x[None, :], th[:, :1], th[:, 1:])
    assert common.rel_err(pw, want_pw) < TOL_PW
    # each observation is its own problem: the chunked call gives the bits of one call per slice
    for a, b in ((0, 2047), (2047, n_obs))[: 1 if n_obs == 2047 else 2]:
        with bound("gaussian", dict(x=x[a:b]), 2) as h:
            assert np.array_equal(np.array(h.loo(th)), got[:, a:b], equal_nan=True)
    idx = [0, 2046, n_obs - 1]
    want = ref_loo(pw.T[idx])
    for q in range(4):
        assert abs_err(got[q][idx], want[q]) < TOL_LOO


@pytest.mark.parametrize("devices", [[0, 1], [0, 1, 2]])
def test_multi_device_slices_give_the_same_bits(loo_emu, devices):
    # each device takes a contiguous slice of the observations and writes it at its offset
    rng = np.random.default_rng(9)
    kw, d, draws, _ = model_case("lba", rng, 101)
    th = draws(50)
    with bound("lba", kw, d) as h:
        one, pw1, part1 = np.array(h.loo(th)), h.eval_pointwise(th), h.eval_pointwise(th, obs0=17, n_obs=40)
    with bound("lba", kw, d, devices=devices) as h:
        many, pwn, partn = np.array(h.loo(th)), h.eval_pointwise(th), h.eval_pointwise(th, obs0=17, n_obs=40)
    assert np.array_equal(one, many, equal_nan=True) and np.array_equal(pw1, pwn) and np.array_equal(part1, partn)


def test_api_on_chains(loo_emu):
    rng = np.random.default_rng(2)
    x = rng.normal(0, 1, 30)
    model = D.DEModel(sample_prior=lambda: [rng.normal(), 1.0], loglike=D.GPULoglike("gaussian", x), names=("mu", "sigma"))
    v = np.zeros((50, 4, 6))
    v[:, 0, :] = rng.normal(0, 0.2, (50, 6))
    v[:, 1, :] = rng.uniform(0.8, 1.2, (50, 6))
    chains = D.Chains(v, ["mu", "sigma", "acceptance", "lp"], ["mu", "sigma"])
    pw = D.pointwise_loglikelihoods(model, chains)
    assert pw.shape == (30, 50, 6)
    assert np.array_equal(pw[:, 7, 3], st.norm.logpdf(x, v[7, 0, 3], v[7, 1, 3])) or \
        common.rel_err(pw[:, 7, 3], st.norm.logpdf(x, v[7, 0, 3], v[7, 1, 3])) < TOL_PW
    r = D.loo(model, chains)
    ll = pw.reshape(30, -1)
    want = ref_loo(ll)
    assert abs_err(r["elpd_loo_i"], want[0]) < TOL_LOO and abs_err(r["pareto_k"], want[1]) < TOL_LOO
    assert math.isclose(r["elpd_loo"], want[0].sum(), rel_tol=1e-12)
    assert math.isclose(r["p_loo"], want[2].sum() - want[0].sum(), rel_tol=1e-9, abs_tol=1e-11)
    assert math.isclose(r["elpd_waic"], (want[2] - want[3]).sum(), rel_tol=1e-12)
    assert math.isclose(r["se_elpd_loo"], math.sqrt(30 * np.var(want[0])), rel_tol=1e-9)
    assert r["n_bad_k"] == int(np.sum(want[1] > 0.7))


# ---- GPU ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_gpu_pointwise_at_1e5(cuda, kind):
    check_pointwise(kind, 100_000, 8)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["gaussian", "lnr", "lba"])
def test_gpu_custom_sources_match_the_registered_kernels(cuda, kind):
    from test_custom_loglike import GAUSS, LBA, LNR
    rng = np.random.default_rng(21)
    kw, d, draws, _ = model_case(kind, rng, 5000)
    th = draws(40)
    with bound(kind, kw, d) as h:
        want = h.eval_pointwise(th)
    x = kw["x"] if kind == "gaussian" else np.column_stack([kw["x"], kw["choice"].astype(float)])
    with bound("custom", dict(x=x, source={"gaussian": GAUSS, "lnr": LNR, "lba": LBA}[kind]), d) as h:
        got = h.eval_pointwise(th)
        part = h.eval_pointwise(th, obs0=1234, n_obs=77)
    assert common.rel_err(got, want) < TOL_PW
    assert np.array_equal(part, got[:, 1234:1311])


def lba_posterior_draws(rng, S):
    return np.column_stack([rng.normal([3, 2], 0.05, (S, 2)), rng.normal(0.8, 0.01, S), rng.normal(0.2, 0.01, S),
                            rng.uniform(0.28, 0.3, S)])


@pytest.mark.gpu
@pytest.mark.parametrize("S, n", [(4000, 100_000), (16384, 3000)])
def test_gpu_loo_matches_the_reference(cuda, S, n):
    # configs[2]'s shape (LBA, 2 accumulators, 1e5 trials) at S = 4000, and the cap; the reference runs on 300 observations:
    # the ones with the largest k-hat, the smallest, and a spread of the rest
    rng = np.random.default_rng(88484)
    choice, rt = lba_vec(rng, n)
    th = lba_posterior_draws(rng, S)
    with bound("lba", dict(x=rt, choice=choice, n_dim=2), 5) as h:
        got = np.array(h.loo(th))
        again = np.array(h.loo(th))
        order = np.argsort(got[1])
        idx = np.unique(np.concatenate([order[:50], order[-150:], np.linspace(0, n - 1, 100).astype(int)]))
        ll = np.stack([h.eval_pointwise(th, obs0=int(i), n_obs=1)[:, 0] for i in idx])
    assert np.array_equal(got, again, equal_nan=True)
    want = ref_loo(ll)
    for q in range(4):
        assert abs_err(got[q][idx], want[q]) < TOL_LOO, q


@pytest.mark.gpu
def test_gpu_conjugate_model_end_to_end(cuda):
    # a one-parameter custom source, sample(), then loo(): within a few Monte-Carlo standard errors of the exact elpd_loo
    y, _, exact, tau = conjugate()
    src = """
__device__ double demcmc_obs(const double *th, const double *x)
{
    const double z = x[0] - th[0];
    return -(z * z + 1.8378770664093454836) / 2.0;
}
"""
    rng = np.random.default_rng(12)
    model = D.DEModel(sample_prior=lambda: [rng.normal(0, tau)], prior_loglike=D.GPUPrior(D.Normal(0, tau)),
                      loglike=D.GPULoglike("custom", y, source=src), names=("mu",))
    de = D.DE(sample_prior=model.sample_prior, bounds=((-np.inf, np.inf),), burnin=1000, Np=8, n_groups=4, seed=31)
    chains = D.sample(model, de, D.MCMCThreads(), 1500)
    assert chains.value.shape[0] * chains.value.shape[2] == 16000
    r = D.loo(model, chains)
    # thinned to about independent draws the same check as on exact draws: 4 Monte-Carlo SE + the MCMC error of elpd
    assert abs(r["elpd_loo"] - exact) < 0.1, (r["elpd_loo"], exact)
    assert r["n_bad_k"] == 0 and r["p_loo"] > 0.5 and r["p_loo"] < 1.5


@pytest.mark.gpu
def test_gpu_outlier_has_the_largest_k(cuda):
    rng = np.random.default_rng(3)
    y = np.concatenate([rng.normal(0, 1, 99), [15.0]])
    model = D.DEModel(sample_prior=lambda: [rng.normal(), abs(rng.normal()) + 0.5], prior_loglike=D.GPUPrior(D.Normal(0, 5), D.HalfCauchy(0, 1)),
                      loglike=D.GPULoglike("gaussian", y), names=("mu", "sigma"))
    de = D.DE(sample_prior=model.sample_prior, bounds=((-np.inf, np.inf), (0.0, np.inf)), burnin=1000, Np=8, n_groups=4, seed=7)
    chains = D.sample(model, de, D.MCMCThreads(), 1500)
    r = D.loo(model, chains)
    assert int(np.argmax(r["pareto_k"])) == 99 and r["pareto_k"][99] > 0.7, r["pareto_k"][95:]


@pytest.mark.gpu
def test_gpu_two_devices_give_the_same_bits(cuda):
    if D._ffi.lib().demcmc_device_count() < 2:
        pytest.skip("one GPU")
    rng = np.random.default_rng(6)
    kw, d, draws, _ = model_case("lba", rng, 20_001)
    th = draws(1000)
    with bound("lba", kw, d) as h:
        one, pw1 = np.array(h.loo(th)), h.eval_pointwise(th)
    with bound("lba", kw, d, devices=[0, 1]) as h:
        two, pw2 = np.array(h.loo(th)), h.eval_pointwise(th)
    assert np.array_equal(one, two, equal_nan=True) and np.array_equal(pw1, pw2)

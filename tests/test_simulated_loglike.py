"""Simulation-based likelihoods: GPULoglike("simulated", X, source=..., n_sim=M) estimates each proposal's density from M
simulations of a user-written simulator (include/demcmc_b200.h: DEMCMC_SIMULATED).

CPU part: the NVRTC compile step (no device needed), the argument checks, the host-only test double's refusal, and an
extended-precision numpy reference of the estimator, itself checked against scipy.stats.gaussian_kde and numpy's quantile
and sd.  GPU part: the random streams, the estimator against that reference on the simulations the device returns, the
likelihood every traced proposal of a run got, the pointwise / LOO path, two posteriors next to the registered kernels,
and determinism, rebinding, the compile cache and a two-device handle."""
import time

import numpy as np
import pytest
import scipy.stats as st

import common
from common import D

SWEEP_EVAL = 0xFFFFFFFF

GAUSS_SIM = """
// Normal(mu, sigma): theta = {mu, sigma}
__device__ void demcmc_simulate(const double *th, demcmc_rng *rng, double *y) { y[0] = th[0] + th[1] * demcmc_normal(rng); }
"""
# 2-accumulator LBA (Brown & Heathcote 2008), drift sd 1: theta = {v1, v2, A, k, tau}; y = {choice, rt}.  The drifts are
# redrawn until one is positive, as common.lba_sim does: the registered kernel's density is conditional on a response.
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
UNIFORM_SIM = "__device__ void demcmc_simulate(const double *th, demcmc_rng *rng, double *y) { y[0] = demcmc_uniform(rng); }\n"
NORMAL_SIM = "__device__ void demcmc_simulate(const double *th, demcmc_rng *rng, double *y) { y[0] = demcmc_normal(rng); }\n"


# ---- the reference of DEMCMC_SIMULATED steps 2-5, in extended precision ------------------------------------------------
L = np.longdouble


def quantile_linear(v, p):
    """Linearly interpolated quantile of sorted v (numpy's default method), in long double."""
    h = L(len(v) - 1) * L(p)
    lo = int(np.floor(h))
    hi = min(lo + 1, len(v) - 1)
    return v[lo] + (h - L(lo)) * (v[hi] - v[lo])


def silverman(vals):
    """h of one group (long double), or None when the group has no density."""
    m = len(vals)
    if m < 2:
        return None
    v = np.sort(np.asarray(vals, dtype=L))
    mean = v.sum() / L(m)
    s = np.sqrt(((v - mean) ** 2).sum() / L(m - 1))
    iqr = quantile_linear(v, 0.75) - quantile_linear(v, 0.25)
    a = min(s, iqr / L(1.34)) if iqr > 0 else s
    h = L(0.9) * a * L(m) ** L(-0.2)
    return h if (h > 0 and np.isfinite(h)) else None


def groups(sims, n_cols):
    """label -> the finite values of the simulations with exactly that label (n_cols = 1: label 1)."""
    val = sims[:, -1]
    fin = np.isfinite(val)
    if n_cols == 1:
        return {1: val[fin]}
    lab = sims[:, 0]
    return {c: val[fin & (lab == c)] for c in range(1, 9)}


def reference_ll(sims, x, floor):
    """ll_i (long double) of the observations x[N] (n_cols = 1) or x[N][2] for the simulations sims[M][n_cols]."""
    sims = np.asarray(sims, dtype=np.float64).reshape(len(sims), -1)
    n_cols = sims.shape[1]
    M = len(sims)
    x = np.asarray(x, dtype=np.float64).reshape(-1, n_cols)
    g = groups(sims, n_cols)
    out = np.full(len(x), np.log(L(floor)), dtype=L)
    labels = np.ones(len(x), dtype=int) if n_cols == 1 else x[:, 0].astype(int)
    for c in np.unique(labels):
        vals = g.get(c, np.zeros(0))
        h = silverman(vals)
        if h is None:
            continue
        idx = np.nonzero(labels == c)[0]
        v = np.asarray(vals, dtype=L)
        for a in range(0, len(idx), 256):
            ii = idx[a:a + 256]
            z = (x[ii, -1].astype(L)[:, None] - v[None, :]) / h
            f = np.exp(-z * z / 2).sum(axis=1) / (np.sqrt(2 * L(np.pi)) * L(M) * h)
            out[ii] = np.log(np.maximum(f, L(floor)))
    return out


class TestReference:
    """The reference on its own, against scipy / numpy (float64 implementations of the same quantities)."""

    def test_bandwidth_is_silverman_from_numpy_quantile_and_sd(self):
        rng = np.random.default_rng(3)
        for m in (2, 3, 17, 1000):
            v = rng.gamma(2.0, 1.5, m)
            q75, q25 = np.quantile(v, [0.75, 0.25])
            s = np.std(v, ddof=1)
            iqr = q75 - q25
            h = 0.9 * (min(s, iqr / 1.34) if iqr > 0 else s) * m ** -0.2
            assert abs(float(silverman(v)) - h) <= 1e-13 * h
        # IQR = 0 with s > 0 uses s alone; a constant group and a single simulation have no density
        v = np.array([0.0] * 10 + [5.0])
        assert abs(float(silverman(v)) - 0.9 * np.std(v, ddof=1) * 11 ** -0.2) <= 1e-13
        assert silverman(np.full(7, 2.5)) is None and silverman(np.array([1.0])) is None and silverman(np.zeros(0)) is None

    def test_density_is_gaussian_kde_at_the_same_bandwidth_scaled_by_the_group_share(self):
        rng = np.random.default_rng(5)
        M = 400
        sims = np.column_stack([rng.integers(1, 3, M).astype(float), rng.lognormal(-0.5, 0.4, M)])
        sims[:7, 1] = np.nan                                       # outside every group, still counted in M
        sims[7:12, 0] = 3.5                                        # not an integer label: no group
        x = np.column_stack([rng.integers(1, 3, 50).astype(float), rng.lognormal(-0.5, 0.5, 50)])
        ref = reference_ll(sims, x, 1e-300)
        g = groups(sims, 2)
        for c in (1, 2):
            v = g[c]
            h = float(silverman(v))
            kde = st.gaussian_kde(v, bw_method=h / np.std(v, ddof=1))
            sel = x[:, 0] == c
            f = kde(x[sel, 1]) * len(v) / M
            assert np.allclose(np.exp(ref[sel].astype(float)), f, rtol=1e-10, atol=0)

    def test_floor_and_empty_groups(self):
        sims = np.column_stack([np.ones(32), np.linspace(0.2, 0.8, 32)])
        x = np.array([[1.0, 0.5], [1.0, 1e6], [2.0, 0.5]])       # in range; far from every simulation; never simulated
        ref = reference_ll(sims, x, 1e-10)
        assert ref[0] > np.log(1e-10)
        assert ref[1] == np.log(L(1e-10)) and ref[2] == np.log(L(1e-10))


# ---- CPU: compile step, argument checks, the test double ------------------------------------------------------------
@pytest.mark.usefixtures("cuda")
class TestCompile:
    def test_accepts_sources_with_and_without_prepare(self):
        D.handle.compile_simulator(GAUSS_SIM)
        D.handle.compile_simulator(LBA_SIM)

    def test_syntax_error_names_user_cu_and_the_line(self):
        with pytest.raises(D._ffi.DemcmcError) as e:
            D.handle.compile_simulator("__device__ void demcmc_simulate(const double *p, demcmc_rng *r, double *y)\n{\n    y[0] = ;\n}\n")
        assert e.value.code == -1
        assert "user.cu(3)" in str(e.value), str(e.value)

    def test_missing_simulate_is_named(self):
        with pytest.raises(D._ffi.DemcmcError) as e:
            D.handle.compile_simulator("__device__ double helper(double a) { return a; }\n")
        assert e.value.code == -1 and "demcmc_simulate" in str(e.value)

    def test_npar_above_the_cap_is_unsupported(self):
        with pytest.raises(D._ffi.DemcmcError) as e:
            D.handle.compile_simulator("#define DEMCMC_NPAR 300\n__device__ void demcmc_prepare(const double *t, double *p) {}\n" + GAUSS_SIM)
        assert e.value.code == -6

    def test_a_custom_source_of_the_same_text_is_cached_apart(self):
        # the same text is a valid simulator and an invalid custom likelihood: each cache entry keeps its own verdict
        D.handle.compile_simulator(GAUSS_SIM)
        with pytest.raises(D._ffi.DemcmcError, match="demcmc_obs"):
            D.handle.compile_loglike(GAUSS_SIM)
        D.handle.compile_simulator(GAUSS_SIM)

    def test_gpuloglike_checks_its_arguments(self):
        x2 = np.column_stack([np.ones(5), np.linspace(0.3, 0.9, 5)])
        with pytest.raises(ValueError, match="n_cols"):
            D.GPULoglike("simulated", np.zeros((5, 3)), source=GAUSS_SIM, n_sim=64)
        bad = x2.copy(); bad[2, 0] = 1.5
        with pytest.raises(ValueError, match="labels must be integers in 1..8"):
            D.GPULoglike("simulated", bad, source=LBA_SIM, n_sim=64)
        bad[2, 0] = 9.0
        with pytest.raises(ValueError, match="labels must be integers in 1..8"):
            D.GPULoglike("simulated", bad, source=LBA_SIM, n_sim=64)
        bad = x2.copy(); bad[1, 1] = np.inf
        with pytest.raises(ValueError, match="finite"):
            D.GPULoglike("simulated", bad, source=LBA_SIM, n_sim=64)
        for m in (None, 15, 16385):
            with pytest.raises(ValueError, match="n_sim"):
                D.GPULoglike("simulated", x2, source=LBA_SIM, n_sim=m)
        for f in (0.0, -1e-10):
            with pytest.raises(ValueError, match="floor"):
                D.GPULoglike("simulated", x2, source=LBA_SIM, n_sim=64, floor=f)
        with pytest.raises(ValueError, match="source"):
            D.GPULoglike("simulated", x2, n_sim=64)
        with pytest.raises(D._ffi.DemcmcError, match="user.cu"):
            D.GPULoglike("simulated", x2, source="__device__ void demcmc_simulate(const double *p, demcmc_rng *r, double *y) { y[0] = }", n_sim=64)
        ll = D.GPULoglike("simulated", x2, source=LBA_SIM, n_sim=64)
        assert ll.kind == "simulated" and ll.n_sim == 64 and ll.sim_floor == 1e-10


@pytest.mark.usefixtures("emu")
def test_the_test_double_refuses_simulated_models():
    with D.Handle(2, 4, 2, [-np.inf, 0.0], [np.inf, np.inf]) as h:
        with pytest.raises(D._ffi.DemcmcError) as e:
            h.set_model("simulated", [("flat",)] * 2, x=np.zeros(10), source=GAUSS_SIM, n_sim=64)
    assert e.value.code == -6 and "simulated likelihoods need the CUDA backend" in str(e.value)


# ---- GPU ----------------------------------------------------------------------------------------------------------
def _handle(d, x, src, n_sim, floor=1e-10, **kw):
    h = D.Handle(4, 8, d, [-np.inf] * d, [np.inf] * d, **kw)
    h.set_model("simulated", [("flat",)] * d, x=x, source=src, n_sim=n_sim, sim_floor=floor)
    return h


def _lba_theta(rng, n):
    return np.column_stack([rng.uniform(1.5, 3.5, n), rng.uniform(0.5, 2.5, n), rng.uniform(0.3, 1.0, n),
                            rng.uniform(0.1, 0.5, n), rng.uniform(0.1, 0.3, n)])


def _rel(dev, ref):
    """|dev - ref| relative to sum_i |ll_i| of the reference."""
    return float(abs(L(dev) - ref.sum()) / max(L(1), np.abs(ref).sum()))


# worst relative error of the device's log-likelihood against the reference, measured on one B200; tolerance 100x
PARITY_WORST = 9.7e-16                                       # LBA, N = 257, M = 17 (Gaussian: 3.5e-16)
PARITY_TOL = 100 * PARITY_WORST


@pytest.mark.gpu
@pytest.mark.usefixtures("cuda")
class TestDevice:
    def test_random_streams(self):
        n, M = 64, 16384                                           # 1 048 576 draws
        for src, cdf in ((UNIFORM_SIM, st.uniform.cdf), (NORMAL_SIM, st.norm.cdf)):
            with _handle(1, np.zeros(4), src, M, seed=77) as h:
                sweep, unit = np.arange(n, dtype=np.uint32) * 3, np.arange(n, dtype=np.uint32) + 1000
                _, s1 = h.eval_simulated(np.zeros((n, 1)), sweep, unit, sims=True)
                _, s2 = h.eval_simulated(np.zeros((n, 1)), sweep, unit, sims=True)
                assert np.array_equal(s1, s2)
                draws = s1.reshape(-1)
                assert st.kstest(draws, cdf).pvalue > 1e-3
                if src is UNIFORM_SIM:
                    assert draws.min() > 0.0 and draws.max() < 1.0
                _, other_sweep = h.eval_simulated(np.zeros((n, 1)), sweep + 1, unit, sims=True)
                _, other_unit = h.eval_simulated(np.zeros((n, 1)), sweep, unit + 1, sims=True)
                assert not np.any(other_sweep == s1) and not np.any(other_unit == s1)
            with _handle(1, np.zeros(4), src, M, seed=78) as h:
                _, other_seed = h.eval_simulated(np.zeros((n, 1)), sweep, unit, sims=True)
                assert not np.any(other_seed == s1)

    @pytest.mark.parametrize("n_obs", [1, 255, 257, 10_000])
    @pytest.mark.parametrize("model", ["gaussian", "lba"])
    def test_estimator_matches_the_reference(self, model, n_obs):
        self._parity(model, n_obs, 512)

    @pytest.mark.parametrize("M", [17, 1000])
    @pytest.mark.parametrize("model", ["gaussian", "lba"])
    def test_simulation_counts_that_are_not_a_power_of_two(self, model, M):
        # the sort pads the M simulations to a power of two with entries in no group; at M = 17 some LBA label groups
        # have fewer than two simulations and no density
        self._parity(model, 257, M)

    def _parity(self, model, n_obs, M):
        rng = np.random.default_rng(600 + n_obs + M)
        if model == "gaussian":
            x, src, d = rng.normal(0.3, 1.2, n_obs), GAUSS_SIM, 2
            th = np.column_stack([rng.normal(0.3, 0.3, 64), rng.uniform(0.6, 2.0, 64)])
        else:
            c, rt = common.lba_sim(rng, n_obs)
            x, src, d = np.column_stack([c.astype(float), rt]), LBA_SIM, 5
            th = _lba_theta(rng, 64)
        with _handle(d, x, src, M) as h:
            keys = rng.integers(0, 2**32 - 1, (2, 64), dtype=np.uint64).astype(np.uint32)
            ll, sims = h.eval_simulated(th, keys[0], keys[1], sims=True)
        worst = max(_rel(ll[i], reference_ll(sims[i], x, 1e-10)) for i in range(64))
        print(f"simulated {model} N={n_obs} M={M}: worst relative error {worst:.3g}")
        assert worst <= PARITY_TOL, worst

    def test_floor_cases(self):
        rng = np.random.default_rng(9)
        # label 3 is never simulated by a 2-accumulator simulator; rt 1e6 is far from every simulation
        x = np.array([[1.0, 0.6], [2.0, 0.7], [1.0, 1e6], [3.0, 0.6]])
        with _handle(5, x, LBA_SIM, 256, floor=1e-7) as h:
            th = _lba_theta(rng, 8)
            ll, sims = h.eval_simulated(th, np.zeros(8), np.arange(8), sims=True)
            pw = h.eval_pointwise(th)
        for i in range(8):
            ref = reference_ll(sims[i], x, 1e-7)
            assert abs(ll[i] - float(ref.sum())) <= PARITY_TOL * float(np.abs(ref).sum())
        assert np.all(pw[:, 2] == np.log(1e-7)) and np.all(pw[:, 3] == np.log(1e-7))

    @pytest.mark.parametrize("kw", [dict(theta_snooker=0.1, alpha=0.3), dict(blocks=np.array([[1, 1, 0, 0, 0], [0, 0, 1, 1, 1]], np.uint8))],
                             ids=["snooker_migration", "blocked"])
    def test_the_run_computes_the_estimator(self, kw):
        rng = np.random.default_rng(21)
        c, rt = common.lba_sim(rng, 300)
        x = np.column_stack([c.astype(float), rt])
        prior = [("normal", 2.0, 3.0), ("normal", 2.0, 3.0), ("normal", 0.8, 0.4), ("normal", 0.3, 0.3), ("normal", 0.2, 0.1)]
        lo, hi = [0.0, 0.0, 0.05, 0.01, 0.0], [10.0, 10.0, 2.0, 2.0, 0.29]
        with D.Handle(4, 8, 5, lo, hi, burnin=5, seed=31, trace=True, **kw) as h:
            h.set_model("simulated", prior, x=x, source=LBA_SIM, n_sim=256)
            h.set_state(_lba_theta(rng, 32))
            h.run(12)                                              # with alpha < 1, chunks of several sweeps
            tr = h.trace()
            S = tr["prop_weight"].shape[0]
            assert S == 12 * h.B
            th = tr["prop_theta"].reshape(-1, 5)
            sweep = np.repeat(np.arange(S, dtype=np.uint32), 32)
            unit = np.tile(np.arange(32, dtype=np.uint32), S)     # one group block: global position = local position
            ll = h.eval_simulated(th, sweep, unit)
            _, pr = h.eval(th)
        expect = (pr + ll).reshape(S, 32)
        assert np.array_equal(tr["prop_weight"], expect, equal_nan=True)
        assert np.isfinite(tr["prop_weight"]).mean() > 0.5

    def test_the_library_checks_its_arguments(self):
        x2 = np.column_stack([np.ones(5), np.linspace(0.3, 0.9, 5)])
        with D.Handle(2, 4, 2, [-np.inf, 0.0], [np.inf, np.inf]) as h:
            for bad, msg in ((dict(x=np.zeros((5, 3))), "n_cols"), (dict(x=x2, n_sim=15), "n_sim"), (dict(x=x2, n_sim=16385), "n_sim"),
                             (dict(x=x2, sim_floor=0.0), "sim_floor"), (dict(x=x2, source=None), "source"),
                             (dict(x=np.column_stack([np.full(5, 9.0), x2[:, 1]])), "label"),
                             (dict(x=np.column_stack([np.full(5, 1.5), x2[:, 1]])), "label"),
                             (dict(x=np.array([0.1, np.nan])), "finite")):
                kw = dict(source=GAUSS_SIM, n_sim=64) | bad
                with pytest.raises(D._ffi.DemcmcError, match=msg) as e:
                    h.set_model("simulated", [("flat",)] * 2, **kw)
                assert e.value.code == -1
            import torch
            xd = torch.zeros(10, dtype=torch.float64, device="cuda")
            with pytest.raises(D._ffi.DemcmcError, match="host data") as e:
                h.set_model("simulated", [("flat",)] * 2, device_ptrs=(xd.data_ptr(), None), n_obs=10, n_cols=1, source=GAUSS_SIM, n_sim=64)

    def test_pointwise_and_loo(self):
        rng = np.random.default_rng(33)
        c, rt = common.lba_sim(rng, 700)
        x = np.column_stack([c.astype(float), rt])
        th = _lba_theta(rng, 40)
        with _handle(5, x, LBA_SIM, 512) as h:
            pw = h.eval_pointwise(th)
            ll, _ = h.eval(th)
            _, sims = h.eval_simulated(th, np.full(40, SWEEP_EVAL, np.uint32), np.arange(40), sims=True)
            elpd, k, lppd, p_waic = h.loo(th)
        assert np.allclose(pw.sum(axis=1), ll, rtol=1e-12, atol=0)
        for j in range(40):
            ref = reference_ll(sims[j], x, 1e-10).astype(float)
            assert np.allclose(pw[j], ref, rtol=PARITY_TOL, atol=PARITY_TOL)
        assert np.all(np.isfinite(elpd)) and np.all(lppd >= elpd - 1e-12)
        # sample() -> loo() on a simulated model, twice: the same numbers
        res = []
        for _ in range(2):
            r2 = np.random.default_rng(5)
            model = D.DEModel(sample_prior=lambda: [r2.normal(0.3, 0.3), r2.uniform(0.6, 1.5)],
                              prior_loglike=D.GPUPrior(D.Normal(0, 2), D.HalfCauchy(0, 1)),
                              loglike=D.GPULoglike("simulated", rng.__class__(np.random.PCG64(3)).normal(0.3, 1.0, 300), source=GAUSS_SIM, n_sim=256),
                              names=("mu", "sigma"))
            de = D.DE(sample_prior=model.sample_prior, bounds=((-np.inf, np.inf), (0.0, np.inf)), Np=8, n_groups=4, burnin=100, seed=8)
            chains = D.sample(model, de, 300)
            res.append(D.loo(model, chains))
        assert repr(res[0]) == repr(res[1])

    def test_gaussian_posterior_next_to_the_registered_kernel(self):
        rng = np.random.default_rng(500)
        x = rng.normal(0.5, 1.0, 500)
        M = 8192
        out = {}
        for kind in ("gaussian", "simulated"):
            r2 = np.random.default_rng(7)
            ll = D.GPULoglike("gaussian", x) if kind == "gaussian" else D.GPULoglike("simulated", x, source=GAUSS_SIM, n_sim=M)
            model = D.DEModel(sample_prior=lambda: [r2.normal(0.5, 0.2), r2.uniform(0.7, 1.3)],
                              prior_loglike=D.GPUPrior(D.Normal(0, 10), D.HalfCauchy(0, 5)), loglike=ll, names=("mu", "sigma"))
            de = D.DE(sample_prior=model.sample_prior, bounds=((-np.inf, np.inf), (0.0, np.inf)), Np=8, n_groups=32, burnin=300, seed=19)
            ch = D.sample(model, de, 1300)
            out[kind] = (ch.mean()[:2], ch.std()[:2], ch.ess()[:2])
        (m_r, s_r, e_r), (m_s, s_s, e_s) = out["gaussian"], out["simulated"]
        infl = np.sqrt(1 + 0.81 * M ** -0.4)                         # the KDE's variance inflation: h ~ 0.9 sigma M^(-1/5)
        mcse = lambda s, e: s / np.sqrt(e)                          # noqa: E731
        print("registered", m_r, s_r, e_r, "simulated", m_s, s_s, e_s)
        assert abs(m_s[0] - m_r[0]) <= 0.5 * s_r[0] + 3 * np.hypot(mcse(s_r[0], e_r[0]), mcse(s_s[0], e_s[0]))
        assert abs(m_s[1] * infl - m_r[1]) <= 0.5 * s_r[1] + 3 * np.hypot(mcse(s_r[1], e_r[1]), infl * mcse(s_s[1], e_s[1]))

    def test_lba_posterior_next_to_the_registered_kernel(self):
        # 500 trials of a 2-accumulator LBA; the simulated model (M = 8192, the simulator redraws the drifts until one is
        # positive, so its labels' defective densities add up to the registered kernel's density conditional on a response)
        # and the registered LBA kernel on the same data, priors, bounds, seed and start
        rng = np.random.default_rng(510)
        choice, rt = common.lba_sim(rng, 500)
        mn = float(rt.min())
        out = {}
        for kind in ("lba", "simulated"):
            r2 = np.random.default_rng(8)
            ll = (D.GPULoglike("lba", choice=choice, rt=rt) if kind == "lba" else
                  D.GPULoglike("simulated", np.column_stack([choice.astype(float), rt]), source=LBA_SIM, n_sim=8192))
            model = D.DEModel(sample_prior=lambda: [r2.uniform(2.0, 3.5, 2), r2.uniform(0.5, 1.0), r2.uniform(0.1, 0.3), r2.uniform(0.2, 0.95 * mn)],
                              prior_loglike=D.GPUPrior(D.Normal(2.0, 3.0), D.Normal(0.8, 0.4), D.Normal(0.2, 0.2), D.Uniform(0.0, mn)),
                              loglike=ll, names=("v", "A", "k", "tau"))
            de = D.DE(sample_prior=model.sample_prior, bounds=((0.0, np.inf), (0.01, np.inf), (0.01, np.inf), (0.0, mn)), Np=8, n_groups=32,
                      burnin=500, seed=23)
            ch = D.sample(model, de, 2000)
            out[kind] = (ch.mean()[:5], ch.std()[:5], ch.ess()[:5])
        (m_r, s_r, e_r), (m_s, s_s, e_s) = out["lba"], out["simulated"]
        diff = np.abs(m_s - m_r) / s_r
        mcse = np.hypot(s_r / np.sqrt(e_r), s_s / np.sqrt(e_s)) / s_r
        print("registered", m_r, s_r, e_r, "simulated", m_s, s_s, e_s, "|difference| / registered sd", diff, "MCSE / sd", mcse)
        # Criterion.  Measured on one B200 (the chains are deterministic): |difference| / registered sd = 0.20, 0.45, 0.26 for
        # v1, v2, A and 1.23, 1.82 for k, tau; MCSE below 0.04 sd; posterior sd ratios 0.97 to 1.19.
        # - v1, v2, A: within 0.5 registered sd + 3 MCSE, as for the Gaussian.
        # - k and tau set the leading edge of the RT distributions, which the kernel density smears earlier by about its
        #   bandwidth (h ~ 0.9 sd(RT) m^(-1/5), about 0.02 s here): the estimator's known bias, which is real and not
        #   Monte-Carlo noise (MCSE 0.04 sd).  The fit answers with a later tau and a lower k: within 2.5 registered sd, in
        #   that direction.
        # - every posterior sd within a factor 1.5 of the registered one.
        assert np.all(diff[:3] <= 0.5 + 3 * mcse[:3]), diff
        assert np.all(diff[3:] <= 2.5) and m_s[4] > m_r[4] and m_s[3] < m_r[3], (diff, m_s, m_r)
        assert np.all((s_s / s_r > 1 / 1.5) & (s_s / s_r < 1.5)), s_s / s_r

    def _native(self, x, seed=5, devices=None, rebind=None, src=GAUSS_SIM):
        rng = np.random.default_rng(1)
        with D.Handle(4, 8, 2, [-np.inf, 0.0], [np.inf, np.inf], seed=seed, burnin=10, theta_snooker=0.1, alpha=0.3, devices=devices) as h:
            if rebind is not None:
                h.set_model("simulated", [("normal", 0, 1), ("halfcauchy", 0, 1)], x=x, source=rebind, n_sim=256)
            h.set_model("simulated", [("normal", 0, 1), ("halfcauchy", 0, 1)], x=x, source=src, n_sim=256)
            h.set_state(np.column_stack([rng.normal(size=32), rng.uniform(0.5, 2, 32)]))
            h.run(30)
            return h.samples(), h.lp(), h.accept()

    def test_determinism_rebinding_and_the_compile_cache(self):
        x = np.random.default_rng(8).normal(0.2, 1.3, 2000)
        a, b = self._native(x), self._native(x)
        assert all(np.array_equal(u, v) for u, v in zip(a, b))
        c = self._native(x, seed=6)
        assert not np.array_equal(c[0], a[0])
        shifted = GAUSS_SIM.replace("y[0] = th[0]", "y[0] = 5.0 + th[0]")
        assert all(np.array_equal(u, v) for u, v in zip(self._native(x, rebind=shifted), a))
        fresh = GAUSS_SIM + "\n// %d\n" % time.time_ns()
        with D.Handle(4, 8, 2, [-np.inf, 0.0], [np.inf, np.inf]) as h:
            t0 = time.perf_counter()
            h.set_model("simulated", [("flat",)] * 2, x=x, source=fresh, n_sim=64)
            t1 = time.perf_counter()
            h.set_model("simulated", [("flat",)] * 2, x=x, source=fresh, n_sim=64)
            t2 = time.perf_counter()
        assert t2 - t1 < 0.25 * (t1 - t0), (t1 - t0, t2 - t1)

    def test_multi_device_handle_is_the_single_device_chain(self):
        if D._ffi.lib().demcmc_device_count() < 2:
            pytest.skip("a multi-device handle needs two GPUs")
        x = np.random.default_rng(9).normal(0.2, 1.3, 2000)
        a, b = self._native(x), self._native(x, devices=[0, 1])
        assert all(np.array_equal(u, v) for u, v in zip(a, b))

"""User-written likelihoods: GPULoglike("custom", X, source=...) compiled at run time for sm_100a (include/demcmc_b200.h:
DEMCMC_CUSTOM).

CPU part: the NVRTC compile step (no device needed), the Python argument checks and the host-only test double's refusal.
GPU part: a custom source of a registered density agrees with the registered kernel, densities the library has never
seen agree with scipy / numpy, replayed oracle tapes give the registered kind's accept decisions, and native runs are
deterministic, rebind, hit the compile cache and shard over devices bit for bit."""
import math
import time

import numpy as np
import pytest
import scipy.stats as st

import common
from common import D, forced_run, make_case, rel_err

LOG2PI = "1.8378770664093454836"

# Examples/Gaussian_Example.jl's loglike, written the way the registered kernel evaluates it
GAUSS = """
#define DEMCMC_NPAR 3
__device__ void demcmc_prepare(const double *theta, double *par) { par[0] = theta[0]; par[1] = theta[1]; par[2] = log(theta[1]); }
__device__ double demcmc_obs(const double *par, const double *x)
{
    const double z = (x[0] - par[0]) / par[1];
    return -(z * z + LOG2PI) / 2.0 - par[2];
}
""".replace("LOG2PI", LOG2PI)
GAUSS_PLAIN = """
__device__ double demcmc_obs(const double *th, const double *x)
{
    const double z = (x[0] - th[0]) / th[1];
    return -(z * z + LOG2PI) / 2.0 - log(th[1]);
}
""".replace("LOG2PI", LOG2PI)
# LNR with 4 accumulators, sigma = 1: x = {rt, choice (1-based)}, theta = {nu[4], tau}
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
# LBA with 2 accumulators (Brown & Heathcote 2008, sd 1, density floor 1e-10): x = {rt, choice}, theta = {v1, v2, A, k, tau}
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
# models with no registered kernel
WEIBULL = """
// Weibull(shape k, scale lambda) shifted by s: theta = {k, lambda, s}
#define DEMCMC_NPAR 4
__device__ void demcmc_prepare(const double *th, double *par) { par[0] = th[0]; par[1] = th[1]; par[2] = th[2]; par[3] = log(th[0] / th[1]); }
__device__ double demcmc_obs(const double *par, const double *x)
{
    const double z = (x[0] - par[2]) / par[1];
    if (!(z > 0.0)) return -DEMCMC_INF;
    return par[3] + (par[0] - 1.0) * log(z) - pow(z, par[0]);
}
"""
LOGIT = """
// Bernoulli-logit regression: x = {x1, x2, y}, theta = {b0, b1, b2}
__device__ double demcmc_obs(const double *b, const double *x)
{
    const double eta = b[0] + b[1] * x[0] + b[2] * x[1];
    const double l1pe = eta > 0.0 ? eta + log1p(exp(-eta)) : log1p(exp(eta));
    return x[2] * eta - l1pe;
}
"""
RASTRIGIN = """
// test/optimization_tests.jl:15-23 as an objective of the parameters alone
__device__ double demcmc_particle(const double *x)
{
    double y = 20.0;
    for (int i = 0; i < 2; ++i) y += x[i] * x[i] - 10.0 * cos(2.0 * 3.14159265358979323846 * x[i]);
    return y;
}
"""


def lnr_x(case):
    return np.column_stack([case.data["x"], case.data["choice"].astype(np.float64)])


# ---- CPU: compile step, argument checks, the test double ---------------------------------------------------------
@pytest.mark.usefixtures("cuda")
class TestCompile:
    def test_accepts_gaussian_with_and_without_prepare(self):
        D.handle.compile_loglike(GAUSS)
        D.handle.compile_loglike(GAUSS_PLAIN)
        D.handle.compile_loglike(RASTRIGIN)          # no observations: demcmc_particle alone

    def test_syntax_error_names_user_cu_and_the_line(self):
        with pytest.raises(D._ffi.DemcmcError) as e:
            D.handle.compile_loglike("__device__ double demcmc_obs(const double *p, const double *x)\n{\n    return p[0] + ;\n}\n")
        assert e.value.code == -1
        assert "user.cu(3)" in str(e.value), str(e.value)
        assert "user.cu(3)" in D._ffi.lib().demcmc_last_error().decode()

    def test_missing_obs_is_named(self):
        with pytest.raises(D._ffi.DemcmcError) as e:
            D.handle.compile_loglike("__device__ double helper(double a) { return a; }\n")
        assert e.value.code == -1 and "demcmc_obs" in str(e.value)

    def test_npar_above_the_cap_is_unsupported(self):
        with pytest.raises(D._ffi.DemcmcError) as e:
            D.handle.compile_loglike("#define DEMCMC_NPAR 300\n__device__ void demcmc_prepare(const double *t, double *p) {}\n" + GAUSS_PLAIN)
        assert e.value.code == -6

    def test_gpuloglike_checks_its_arguments(self):
        with pytest.raises(ValueError, match="source"):
            D.GPULoglike("custom", np.zeros(4))
        with pytest.raises(ValueError, match="matrix"):
            D.GPULoglike("custom", np.zeros((2, 3, 4)), source=GAUSS)
        with pytest.raises(ValueError, match="n_cols"):
            D.GPULoglike("custom", np.zeros((5, 0)), source=GAUSS)
        with pytest.raises(D._ffi.DemcmcError, match="user.cu"):
            D.GPULoglike("custom", np.zeros(4), source="__device__ double demcmc_obs(const double *p, const double *x) { return }")
        ll = D.GPULoglike("custom", np.zeros((5, 2)), source=GAUSS)
        assert ll.kind == "custom" and ll.x.shape == (5, 2)


@pytest.mark.usefixtures("emu")
def test_the_test_double_refuses_custom_models():
    with D.Handle(2, 4, 2, [-np.inf, 0.0], [np.inf, np.inf]) as h:
        with pytest.raises(D._ffi.DemcmcError) as e:
            h.set_model("custom", [("flat",)] * 2, x=np.zeros(10), source=GAUSS)
    assert e.value.code == -6 and "custom likelihoods need the CUDA backend" in str(e.value)


# ---- GPU ---------------------------------------------------------------------------------------------------------
def _eval(kind, d, prior, theta, **model):
    with D.Handle(4, 16, d, [-np.inf] * d, [np.inf] * d) as h:
        h.set_model(kind, prior, **model)
        return h.eval(theta)[0]


@pytest.mark.gpu
@pytest.mark.usefixtures("cuda")
class TestDevice:
    def test_agrees_with_the_registered_kernels(self):
        rng = np.random.default_rng(4411)
        n = 100_000
        x = rng.normal(0.3, 1.7, n)
        th = np.column_stack([rng.normal(0, 1, 64), rng.uniform(0.5, 3, 64)])
        pr = [("flat",)] * 2
        ref = _eval("gaussian", 2, pr, th, x=x)
        for src in (GAUSS, GAUSS_PLAIN):
            assert rel_err(_eval("custom", 2, pr, th, x=x, source=src), ref) <= 1e-12
        choice, rt = common.lnr_sim(rng, n)
        th = np.column_stack([rng.normal(-2, 0.5, (64, 4)), rng.uniform(0, rt.min(), 64)])
        pr = [("flat",)] * 5
        ref = _eval("lnr", 5, pr, th, x=rt, choice=choice, n_dim=4)
        got = _eval("custom", 5, pr, th, x=np.column_stack([rt, choice.astype(float)]), source=LNR)
        assert np.max(np.abs(got - ref) / np.abs(ref)) <= 1e-10
        choice, rt = common.lba_sim(rng, n)
        th = np.column_stack([rng.uniform(2, 4, 64), rng.uniform(1, 3, 64), rng.uniform(0.5, 1.0, 64), rng.uniform(0.1, 0.4, 64),
                              rng.uniform(0, rt.min(), 64)])
        ref = _eval("lba", 5, pr, th, x=rt, choice=choice, n_dim=2)
        got = _eval("custom", 5, pr, th, x=np.column_stack([rt, choice.astype(float)]), source=LBA)
        assert np.max(np.abs(got - ref) / np.abs(ref)) <= 1e-10

    @pytest.mark.parametrize("n", [1, 255, 257, 100_000])
    def test_models_without_a_registered_kernel(self, n):
        rng = np.random.default_rng(n)
        k, lam, s = 1.7, 2.0, 0.4
        x = s + lam * rng.weibull(k, n)
        th = np.column_stack([rng.uniform(1.2, 2.5, 64), rng.uniform(1.0, 3.0, 64), rng.uniform(0.0, 0.9 * x.min(), 64)])
        got = _eval("custom", 3, [("flat",)] * 3, th, x=x, source=WEIBULL)
        ref = np.array([math.fsum(st.weibull_min.logpdf(x, c=a, loc=c, scale=b)) for a, b, c in th])
        assert np.max(np.abs(got - ref) / np.abs(ref)) <= 1e-12
        X = rng.normal(size=(n, 2))
        y = (rng.uniform(size=n) < 1.0 / (1.0 + np.exp(-(0.3 + X @ [1.2, -0.7])))).astype(float)
        th = rng.normal(0, 1, (64, 3))
        got = _eval("custom", 3, [("flat",)] * 3, th, x=np.column_stack([X, y]), source=LOGIT)
        eta = th[:, :1] + th[:, 1:2] * X[:, 0] + th[:, 2:3] * X[:, 1]
        ref = np.array([math.fsum(v) for v in y * eta - np.logaddexp(0.0, eta)])
        assert np.max(np.abs(got - ref) / np.abs(ref)) <= 1e-12

    def test_no_observations_only_the_particle_term(self):
        th = np.random.default_rng(3).uniform(-5, 5, (64, 2))
        got = _eval("custom", 2, [("flat",)] * 2, th, x=None, source=RASTRIGIN)
        ref = 20.0 + np.sum(th ** 2 - 10.0 * np.cos(2 * np.pi * th), axis=1)
        assert np.max(np.abs(got - ref) / np.maximum(1.0, np.abs(ref))) <= 1e-12
        with D.Handle(4, 16, 2, [-5.0] * 2, [5.0] * 2) as h:       # observations but no demcmc_obs: refused
            with pytest.raises(D._ffi.DemcmcError, match="demcmc_obs"):
                h.set_model("custom", [("flat",)] * 2, x=np.zeros(10), source=RASTRIGIN)

    @pytest.mark.parametrize("model,kw", [("gaussian", dict(theta_snooker=0.1, alpha=0.3)),
                                          ("lnr", dict(theta_snooker=0.1, alpha=0.3)),
                                          ("gaussian", dict(blocks=np.array([[1, 0], [0, 1]], np.uint8), alpha=0.3))],
                             ids=["gaussian_snooker", "lnr_snooker", "gaussian_blocked"])
    def test_replays_the_oracle_tape_of_the_registered_kind(self, model, kw):
        case = make_case(model, np.random.default_rng(71), n_obs=900)
        src, x = (GAUSS, case.data["x"]) if model == "gaussian" else (LNR, lnr_x(case))

        class Custom(common.Case):
            def handle(self, G, Np, **hkw):
                h = D.Handle(G, Np, self.d, self.lo, self.hi, **hkw)
                h.set_model("custom", self.prior, x=x, source=src)
                return h
        cc = Custom(case.name, case.kind, case.d, case.prior, case.lo, case.hi, case.sample_prior, case.data)
        r, out = forced_run(cc, 3, 8, 12, "replay", burnin=6, **kw)
        rtol = 1e-12 if model == "gaussian" else 1e-10
        assert np.array_equal(out["trace"]["accepted"], r["trace"]["accepted"]), "accept decisions differ"
        assert np.array_equal(out["accept"], r["accept"])
        assert rel_err(out["samples"], r["samples"]) <= 1e-12
        assert rel_err(out["trace"]["prop_weight"], r["trace"]["prop_weight"]) <= rtol
        assert rel_err(out["lp"], r["lp"]) <= rtol

    def test_linear_regression_posterior(self):
        rng = np.random.default_rng(2024)
        n, sigma = 400, 0.5
        X = np.column_stack([np.ones(n), rng.normal(size=n), rng.uniform(-1, 1, n)])
        beta = np.array([0.5, -1.0, 2.0])
        y = X @ beta + rng.normal(0, sigma, n)
        src = """
__device__ double demcmc_obs(const double *b, const double *x)
{
    const double r = (x[3] - (b[0] * x[0] + b[1] * x[1] + b[2] * x[2])) / 0.5;
    return -0.5 * r * r;
}
"""
        model = D.DEModel(sample_prior=lambda: [rng.normal(0, 1, 3)], prior_loglike=D.GPUPrior(D.Flat()),
                          loglike=D.GPULoglike("custom", np.column_stack([X, y]), source=src), names=("β",))
        de = D.DE(sample_prior=model.sample_prior, bounds=((-np.inf, np.inf),), burnin=1000, Np=8, n_groups=4, seed=11)
        chains = D.sample(model, de, 6000)
        cov = sigma ** 2 * np.linalg.inv(X.T @ X)
        bhat = np.linalg.solve(X.T @ X, X.T @ y)
        mean, sd = chains.mean()[:3], chains.std()[:3]
        # 5000 draws x 32 correlated chains: the Monte-Carlo error of the mean is a few percent of the posterior sd
        assert np.all(np.abs(mean - bhat) < 0.1 * np.sqrt(np.diag(cov))), (mean, bhat)
        assert np.allclose(sd, np.sqrt(np.diag(cov)), rtol=0.1), (sd, np.sqrt(np.diag(cov)))

    def test_optimize_custom_rastrigin(self):
        vals = []
        for seed in range(1, 11):
            rng = np.random.default_rng(78454111 + seed)
            model = D.DEModel(sample_prior=lambda: [rng.uniform(-5, 5, 2)], loglike=D.GPULoglike("custom", source=RASTRIGIN), names=("x",))
            de = D.DE(sample_prior=model.sample_prior, bounds=((-5.0, 5.0),), Np=6, n_groups=1, update_particle=D.minimize,
                      evaluate_fitness=D.evaluate_fun, seed=seed)
            vals.append(D.get_optimal(de, model, D.optimize(model, de, 10_000))[1])
        assert sum(abs(v) < 1e-8 for v in vals) >= 2, vals          # the registered Rastrigin's criterion (common.optimize_checks)

    def _native(self, src, x, seed=5, devices=None, rebind=None):
        rng = np.random.default_rng(1)
        with D.Handle(4, 8, 2, [-np.inf, 0.0], [np.inf, np.inf], seed=seed, burnin=10, theta_snooker=0.1, alpha=0.3, devices=devices) as h:
            if rebind is not None:
                h.set_model("custom", [("normal", 0, 1), ("halfcauchy", 0, 1)], x=x, source=rebind)
            h.set_model("custom", [("normal", 0, 1), ("halfcauchy", 0, 1)], x=x, source=src)
            h.set_state(np.column_stack([rng.normal(size=32), rng.uniform(0.5, 2, 32)]))
            h.run(30)
            return h.samples(), h.lp(), h.accept()

    def test_determinism_rebinding_and_the_compile_cache(self):
        x = np.random.default_rng(8).normal(0.2, 1.3, 5000)
        a, b = self._native(GAUSS, x), self._native(GAUSS, x)
        assert all(np.array_equal(u, v) for u, v in zip(a, b))
        # rebinding: the handle runs the second source's kernel (a likelihood twice as large), not the first one's
        doubled = GAUSS.replace("return ", "return 2.0 * (").replace(" - par[2];", " - par[2]);")
        c = self._native(doubled, x, rebind=GAUSS)
        with D.Handle(4, 8, 2, [-np.inf, 0.0], [np.inf, np.inf]) as h:
            th = np.array([[0.1, 1.2], [0.3, 0.9]])
            h.set_model("custom", [("flat",)] * 2, x=x, source=GAUSS)
            l1 = h.eval(th)[0]
            h.set_model("custom", [("flat",)] * 2, x=x, source=doubled)
            assert np.allclose(h.eval(th)[0], 2.0 * l1, rtol=1e-14)
        assert not np.array_equal(c[0], a[0])
        # the compile cache: a source seen before does not compile again
        fresh = GAUSS + "\n// %d\n" % time.time_ns()
        with D.Handle(4, 8, 2, [-np.inf, 0.0], [np.inf, np.inf]) as h:
            t0 = time.perf_counter()
            h.set_model("custom", [("flat",)] * 2, x=x, source=fresh)
            t1 = time.perf_counter()
            h.set_model("custom", [("flat",)] * 2, x=x, source=fresh)
            t2 = time.perf_counter()
        assert t2 - t1 < 0.25 * (t1 - t0), (t1 - t0, t2 - t1)

    def test_multi_device_handle_is_the_single_device_chain(self):
        if D._ffi.lib().demcmc_device_count() < 2:
            pytest.skip("a multi-device handle needs two GPUs")
        x = np.random.default_rng(9).normal(0.2, 1.3, 5000)
        a, b = self._native(GAUSS, x), self._native(GAUSS, x, devices=[0, 1])
        assert all(np.array_equal(u, v) for u, v in zip(a, b))

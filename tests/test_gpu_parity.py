"""GPU parity tests proper (-m gpu): the CUDA kernels, called through the C ABI, against the
oracle on the same seeded inputs.

(a) replay mode: the library consumes the oracle's recorded draws; accept decisions must be
    IDENTICAL, proposals and log-densities within 1e-12 relative (fp64).
(b) native mode: both sides draw from the same Philox map (select_base on sweep-start weights).
Full BASELINE sizes are covered through size-independent properties (sufficient statistics in
extended precision, additivity over observation slices)."""
import json
import os

import numpy as np
import pytest

import common
from common import ALL_MODELS, D, O, compare_run, forced_run, hier_blocks, make_case, rel_err

pytestmark = [pytest.mark.gpu, pytest.mark.usefixtures("cuda")]
RTOL = 1e-12   # north_star: proposals and log-densities within 1e-12 relative in fp64
# LNR / LBA densities are differences of erfc/exp terms: a 1-ulp difference between CUDA's and
# glibc's transcendentals is amplified by that cancellation, so their log-densities get 1e-10
RTOL_W = {"lnr": 1e-10, "lba": 1e-10}
KA = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "reference_known_answers.json")))


def check(r, out, rtol=RTOL, rtol_w=None):
    rtol_w = rtol_w or rtol
    assert np.array_equal(out["trace"]["accepted"], r["trace"]["accepted"]), "accept decisions differ"
    assert np.array_equal(out["accept"], r["accept"])
    assert rel_err(out["trace"]["prop_theta"], r["trace"]["prop_theta"]) <= rtol
    assert rel_err(out["trace"]["prop_weight"], r["trace"]["prop_weight"]) <= rtol_w
    assert rel_err(out["trace"]["log_adj"], r["trace"]["log_adj"]) <= 1e-9
    assert rel_err(out["samples"], r["samples"]) <= rtol
    assert rel_err(out["lp"], r["lp"]) <= rtol_w
    assert np.array_equal(out["state"][2], r["final_id"])
    assert np.array_equal(out["mig"], r["tape"]["mig_slots"])


# ---- the reference's own known-answer vectors, on the device -----------------------------------
def test_device_projection():          # test/utility_tests.jl:71-93
    c = KA["projection"]
    assert np.allclose(D.op_project(c["p1"], c["p2"]), np.array(c["expected_num"]) / c["expected_den"], rtol=1e-15)
    rng = np.random.default_rng(0)
    a, b = rng.normal(size=(2, 1003))
    assert rel_err(D.op_project(a, b), O.project(a, b)) <= RTOL


def test_device_reset():               # test/utility_tests.jl:42-69
    for key in ("reset_vector", "reset_matrix"):
        c = KA[key]
        assert np.array_equal(D.op_reset(c["p1"], c["p2"], c["mask"]), np.array(c["expected"]))


def test_device_particle_algebra():    # test/utility_tests.jl:161-199
    for c in KA["algebra"]["cases"]:
        assert np.allclose(D.op_de_proposal(c["pt"], c["pm"], c["pn"], None, c["g"], 0.0, c["b"]), c["expected"], rtol=1e-15)
    rng = np.random.default_rng(1)
    pt, pm, pn, pb, b = rng.normal(size=(5, 101))
    assert np.array_equal(D.op_de_proposal(pt, pm, pn, pb, 0.77, 0.61, b), O.de_proposal(pt, pm, pn, pb, 0.77, 0.61, b))
    assert np.array_equal(D.op_de_proposal(pt, pm, pn, None, 2.38, 0.0, b), O.de_proposal(pt, pm, pn, None, 2.38, 0.0, b))


def test_device_snooker_and_accept():
    rng = np.random.default_rng(2)
    for d in (2, 6, 51, 1003):
        pt, pz, pm, pn, b = rng.normal(size=(5, d))
        out, adj = D.op_snooker(pt, pz, pm, pn, 1.7, b * 1e-3)
        ref = O.snooker_proposal(pt, pz, pm, pn, 1.7, b * 1e-3)
        assert rel_err(out, ref) <= RTOL
        # d = 1003: norm^(d-1) overflows to Inf on both sides => NaN => always reject (SURVEY hard part 5)
        assert np.isclose(adj, O.adjust_loglike(pt, ref, pz), rtol=1e-10, atol=1e-10, equal_nan=True)
        assert np.isnan(adj) == (d == 1003)
    wp = np.array([-1.0, -3.0, -3.0, -np.inf, -np.inf, -np.inf, 1.0])
    wc = np.array([-2.0, -2.0, -2.0, -2.0, -2.0, -np.inf, 2.0])
    adj = np.array([0.0, 0.0, 0.0, 0.0, 0.0, 0.0, np.nan])
    u = np.array([0.999999, np.exp(-1.0) * (1 - 1e-12), np.exp(-1.0) * (1 + 1e-12), 1e-300, 0.0, 0.0, 0.0])
    exp = [O.accept(*t) for t in zip(wp, wc, adj, u)]
    assert list(D.op_accept(wp, wc, adj, u)) == exp == [True, True, False, False, True, False, False]


def test_device_select_quirks():       # SURVEY hard part 4 (softmax under/overflow fallbacks)
    w = np.array([-5000.0, -5100.0, -4900.0, -5050.0])
    for u in np.linspace(0.01, 0.99, 25):
        b, m = D.op_select(w, float(u))
        assert b == O.select_base(w, float(u)) and m == O.select_particle(w, float(u))[0] == 1
    rng = np.random.default_rng(3)
    for n in (3, 24, 256, 4096):
        w = rng.normal(-3, 2, n)
        for u in rng.uniform(size=6):
            b, m = D.op_select(w, float(u))
            assert b == O.select_base(w, float(u)) and m == O.select_particle(w, float(u))[0]


# ---- whole population steps --------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["replay", "native"])
@pytest.mark.parametrize("model", ALL_MODELS)
def test_population_step_all_models(mode, model):
    case = make_case(model, np.random.default_rng(21))
    r, out = forced_run(case, 3, 8, 30, mode, burnin=15, theta_snooker=0.15, alpha=0.3)
    check(r, out, rtol_w=RTOL_W.get(model))


@pytest.mark.parametrize("mode", ["replay", "native"])
@pytest.mark.parametrize("model", ["gaussian", "lnr", "lba"])
def test_pointwise_models_above_the_fused_size(mode, model):
    """Up to 256 observations a level of a pointwise model is ONE launch (k_level_fused: one warp does the
    proposal, the likelihood and the accept of a particle); above, k_propose / k_ll_pointwise / k_accept.
    The default cases of this file are below that size; these are above it, and the two paths are
    compared with each other at a size both accept."""
    case = make_case(model, np.random.default_rng(71), n_obs=900)
    r, out = forced_run(case, 2, 8, 10, mode, burnin=5, theta_snooker=0.2, alpha=0.3)
    check(r, out)


@pytest.mark.parametrize("model", ["gaussian", "lnr", "lba", "binomial"])
def test_fused_level_kernel_against_the_three_kernel_chain(model, monkeypatch):
    case = make_case(model, np.random.default_rng(73))
    theta0 = case.theta0(np.random.default_rng(9), 3 * 8)
    outs = []
    for no_fused in ("1", "0"):
        monkeypatch.setenv("DEMCMC_NO_FUSED", no_fused)
        h = case.handle(3, 8, seed=12, burnin=8, theta_snooker=0.2, alpha=0.3)
        h.set_state(theta0)
        h.run(25)
        outs.append((h.samples(), h.accept(), h.lp(), h.counters()["kernel_launches"]))
        h.close()
    assert outs[1][3] < outs[0][3] * 0.7                                 # one launch per level instead of three (binomial: two)
    assert np.array_equal(outs[0][1], outs[1][1])                       # accept decisions
    assert np.allclose(outs[0][0], outs[1][0], rtol=1e-9, atol=1e-12)    # the likelihood sums differ in order only
    fin = np.isfinite(outs[0][2])
    assert np.allclose(outs[0][2][fin], outs[1][2][fin], rtol=1e-9, atol=1e-9)


@pytest.mark.parametrize("model,kw", [("gaussian", dict(burnin=8, theta_snooker=0.2, alpha=0.3)), ("lnr", dict(burnin=0, kappa=0.8)),
                                      ("lba", dict(burnin=30, alpha=0.5)), ("binomial", dict(burnin=5)), ("gaussian", dict(burnin=4, resample=True, n_initial=5))])
def test_single_cta_chunk_kernel_is_the_level_by_level_chain(model, kw, monkeypatch):
    """A population of a few warps (the reference's own examples) runs every level of a chunk in ONE single-CTA launch
    (k_chunk_small): bit for bit the chain of one k_level_fused launch per level, in a fraction of the launches."""
    rng = np.random.default_rng(79)
    case = make_case(model, rng)
    kw = dict(kw)
    rows = np.stack([case.theta0(rng, 4 * 6) for _ in range(kw["n_initial"])]) if kw.get("resample") else None
    theta0 = case.theta0(np.random.default_rng(9), 4 * 6)
    outs = []
    for no_small in ("1", "0"):
        monkeypatch.setenv("DEMCMC_NO_SMALL", no_small)
        h = case.handle(4, 6, seed=12, **kw)
        if rows is not None:
            h.set_history(rows)
            h.set_state(None)
        else:
            h.set_state(theta0)
        h.run(60)
        outs.append((h.samples(), h.accept(), h.lp(), h.counters()["kernel_launches"]))
        h.close()
    if rows is None:                                          # (DE-MCz donors come from the history: one level per sweep either way)
        assert outs[1][3] < outs[0][3] * 0.6
    for a, b in zip(outs[0][:3], outs[1][:3]):
        assert np.array_equal(a, b, equal_nan=True)


@pytest.mark.parametrize("model", ["gaussian", "mvnormal", "binomial"])
def test_unforced_short_replay(model):
    """Without teacher forcing, over a run short enough that rounding differences are not yet
    amplified by the population dynamics."""
    case = make_case(model, np.random.default_rng(26))
    r, out = compare_run(case, 3, 8, 8, "replay", burnin=4, theta_snooker=0.15, alpha=0.3)
    check(r, out, rtol=1e-11)


@pytest.mark.parametrize("mode", ["replay", "native"])
@pytest.mark.parametrize("kw", [dict(theta_snooker=0.3, kappa=0.8), dict(proposal="fixed_gamma"),
                                dict(proposal="variable_gamma", theta_snooker=0.1), dict(beta=0.5, alpha=0.5)],
                         ids=["snooker_kappa", "fixed_gamma", "variable_gamma", "mutation_migration"])
def test_gaussian_variants(mode, kw):
    case = make_case("gaussian", np.random.default_rng(22))
    r, out = forced_run(case, 4, 6, 100, mode, burnin=50, **kw)
    check(r, out)


@pytest.mark.parametrize("mode", ["replay", "native"])
def test_blocking_hierarchical(mode):   # blocking_on, block masks, last-block-wins (main.jl:174-179)
    case = make_case("hier_normal", np.random.default_rng(23))
    r, out = forced_run(case, 2, 8, 30, mode, burnin=15, blocks=hier_blocks(9), theta_snooker=0.2, alpha=0.3)
    check(r, out)


def test_many_particles_per_group_levels():
    """Np = 256: ~10 dependency levels per sweep must reproduce the sequential in-place sweep."""
    rng = np.random.default_rng(24)
    n, dm = 3000, 50
    x = rng.normal(rng.normal(size=dm), 1.0, size=(n, dm))
    case = common.Case("mvn50", "mvnormal", dm + 1, [("normal", 0, 1)] * dm + [("halfcauchy", 0, 1)], [-np.inf] * dm + [0],
                       [np.inf] * (dm + 1), lambda r: list(r.normal(size=dm)) + [abs(r.standard_cauchy()) + 0.5], dict(x=x))
    r, out = forced_run(case, 2, 256, 4, "replay", burnin=2, theta_snooker=0.1, alpha=0.5)
    check(r, out)
    assert out["counters"]["levels"] >= 4 * 5


def test_ragged_and_tiny_inputs():
    """Observation counts that do not fill a tile, one observation, one dimension."""
    rng = np.random.default_rng(25)
    for n, dm in ((1, 1), (63, 3), (65, 33), (130, 70)):
        x = rng.normal(size=(n, dm))
        case = common.Case("mvn", "mvnormal", dm + 1, [("normal", 0, 1)] * dm + [("halfcauchy", 0, 1)], [-np.inf] * dm + [0],
                           [np.inf] * (dm + 1), lambda r, dm=dm: list(r.normal(size=dm)) + [abs(r.standard_cauchy()) + 0.5], dict(x=x))
        r, out = forced_run(case, 2, 5, 6, "replay", burnin=3, theta_snooker=0.2)
        check(r, out)
    for n in (1, 255, 257, 1000):
        case = make_case("gaussian", np.random.default_rng(n), n_obs=n)
        r, out = forced_run(case, 2, 5, 6, "replay", burnin=3)
        check(r, out)
    # hierarchical with enough subjects for several dimension splits
    S, n = 300, 7
    y = rng.normal(1.0 + rng.normal(0, 1, S)[:, None], 0.5, size=(S, n))
    prior = [("normal", 1, 1), ("halfcauchy", 0, 1)] + [("normal_ref", 0, 0, 1)] * S + [("halfcauchy", 0, 1)]

    def sp(r):
        return [r.normal(1, 1), 1.0] + list(r.normal(0, 1, S)) + [0.7]
    case = common.Case("hier300", "hier_normal", S + 3, prior, [-np.inf, 0] + [-np.inf] * S + [0], [np.inf] * (S + 3), sp, dict(x=y))
    r, out = forced_run(case, 2, 6, 5, "replay", burnin=2, blocks=hier_blocks(S), theta_snooker=0.1)
    check(r, out)


# ---- BASELINE full sizes through size-independent properties -----------------------------------
def test_mvn_full_size_sufficient_statistics():
    """Config 2 shape (d=50, 1e5 obs, 1024 particles): the per-observation kernel must agree with
    the sufficient-statistics identity evaluated in extended precision, and be additive over
    observation slices."""
    rng = np.random.default_rng(50514)
    n, dm, P = 100_000, 50, 1024
    mu = rng.normal(size=dm)
    x = rng.normal(mu, 1.0, size=(n, dm))
    th = np.column_stack([rng.normal(mu, 0.05, size=(P, dm)), rng.uniform(0.8, 1.3, P)])
    prior = [("normal", 0, 1)] * dm + [("halfcauchy", 0, 1)]
    lo, hi = [-np.inf] * dm + [0], [np.inf] * (dm + 1)
    with D.Handle(4, 256, dm + 1, lo, hi) as h:
        h.set_model("mvnormal", prior, x=x)
        ll, _ = h.eval(th)
    xl = x.astype(np.longdouble)
    sx, sxx = xl.sum(axis=0), (xl * xl).sum()
    tl = th.astype(np.longdouble)
    ssd = sxx - 2 * (tl[:, :dm] * sx).sum(axis=1) + n * (tl[:, :dm] ** 2).sum(axis=1)
    ref = -0.5 * n * dm * np.log(2 * np.pi) - n * dm * np.log(tl[:, dm]) - 0.5 * ssd / tl[:, dm] ** 2
    assert np.max(np.abs(ll - ref.astype(float)) / np.abs(ref.astype(float))) <= RTOL
    # additivity over a split of the observations (sizes chosen to leave ragged tiles)
    parts = []
    for sl in (slice(0, 33_333), slice(33_333, n)):
        with D.Handle(4, 256, dm + 1, lo, hi) as h:
            h.set_model("mvnormal", prior, x=x[sl])
            parts.append(h.eval(th)[0])
    assert np.max(np.abs(parts[0] + parts[1] - ll) / np.abs(ll)) <= RTOL


def test_mvn_full_size_posterior_through_the_persistent_kernel():
    """Config 2 at its own size (d=50, 1e5 obs, 4 x 256, crossover + snooker) run natively through the
    persistent chunk kernel: the pooled posterior must sit on the analytic one -- mu_k ~ N(N xbar_k /
    (N + 1), sigma^2 / (N + 1)) given sigma, sigma close to the pooled sd of the centred data -- and the
    device-side moments must agree with the downloaded draws."""
    rng = np.random.default_rng(50514)
    n, dm, G, Np = 100_000, 50, 4, 256
    mu = rng.normal(size=dm)
    x = rng.normal(mu, 1.0, size=(n, dm))
    prior = [("normal", 0, 1)] * dm + [("halfcauchy", 0, 1)]
    lo, hi = [-np.inf] * dm + [0], [np.inf] * (dm + 1)
    xbar = x.mean(axis=0)
    s_pool = np.sqrt(((x - xbar) ** 2).sum() / (n * dm))
    # start near the mode (a cold start needs thousands of iterations at d = 51; this test is about the kernel)
    theta0 = np.column_stack([xbar + rng.normal(0, 1.0 / np.sqrt(n), size=(G * Np, dm)), s_pool * (1 + rng.normal(0, 5e-4, G * Np))])
    n_iter, burn = 700, 300
    with D.Handle(G, Np, dm + 1, lo, hi, seed=77, burnin=0, theta_snooker=0.1) as h:
        h.set_model("mvnormal", prior, x=x)
        h.set_state(theta0)
        h.run(n_iter)
        c = h.counters()
        assert c["persistent_chunks"] > 0
        cnt, mean, var = h.moments(burn, n_iter - burn)
        th = h.history_by_slot(burn, n_iter - burn)[0].reshape(-1, dm + 1)
        acc = h.accept()[:, burn:].mean()
    assert cnt == th.shape[0]
    assert np.allclose(mean, th.mean(axis=0), rtol=1e-12, atol=1e-13) and np.allclose(var, th.var(axis=0, ddof=1), rtol=1e-8)
    assert 0.01 < acc < 0.6, acc
    post_mean = n * xbar / (n + 1.0)
    post_sd = s_pool / np.sqrt(n + 1.0)
    z = (mean[:dm] - post_mean) / post_sd
    assert np.max(np.abs(z)) < 0.6, np.max(np.abs(z))                     # pooled mean of ~1e5 correlated draws
    ratio = np.sqrt(var[:dm]) / post_sd
    assert 0.6 < ratio.min() and ratio.max() < 1.5, (ratio.min(), ratio.max())
    assert abs(mean[dm] / s_pool - 1.0) < 2e-3


def test_lba_full_size_additivity():
    """Config 3 shape (1e5 trials): additivity over trial slices and agreement with the oracle on
    a bounded sample of particles."""
    rng = np.random.default_rng(88484)
    choice, rt = common.lba_sim(rng, 100_000)
    mn = rt.min()
    prior = [("normal", 1, 5), ("normal", 1, 5), ("normal", 0.8, 0.2), ("normal", 0.2, 0.1), ("uniform", 0, mn)]
    lo, hi = [0] * 5, [np.inf] * 4 + [mn]
    th = np.column_stack([rng.uniform(2, 4, 64), rng.uniform(1, 3, 64), rng.uniform(0.5, 1.0, 64), rng.uniform(0.1, 0.4, 64), rng.uniform(0, mn, 64)])
    with D.Handle(4, 16, 5, lo, hi) as h:
        h.set_model("lba", prior, x=rt, choice=choice, n_dim=2)
        ll, _ = h.eval(th)
    m = O.Model("lba", 5, prior, x=rt, choice=choice, n_dim=2)
    ref = np.array([O.loglike(m, t) for t in th[:8]])
    assert np.max(np.abs(ll[:8] - ref) / np.abs(ref)) <= RTOL
    parts = []
    for sl in (slice(0, 41_111), slice(41_111, 100_000)):
        with D.Handle(4, 16, 5, lo, hi) as h:
            h.set_model("lba", prior, x=rt[sl], choice=choice[sl], n_dim=2)
            parts.append(h.eval(th)[0])
    assert np.max(np.abs(parts[0] + parts[1] - ll) / np.abs(ll)) <= RTOL


def test_hier_full_size_against_oracle():
    """Config 4 shape (1000 subjects x 50 obs, d = 1003)."""
    rng = np.random.default_rng(9528)
    S, n = 1000, 50
    y = rng.normal(1.0 + rng.normal(0, 1, S)[:, None], 0.5, size=(S, n))
    prior = [("normal", 1, 1), ("halfcauchy", 0, 1)] + [("normal_ref", 0, 0, 1)] * S + [("halfcauchy", 0, 1)]
    lo, hi = [-np.inf, 0] + [-np.inf] * S + [0], [np.inf] * (S + 3)
    th = np.column_stack([rng.normal(1, 0.1, 40), rng.uniform(0.8, 1.2, 40), rng.normal(0, 1, (40, S)), rng.uniform(0.4, 0.7, 40)])
    with D.Handle(2, 20, S + 3, lo, hi) as h:
        h.set_model("hier_normal", prior, x=y)
        ll, pr = h.eval(th)
    m = O.Model("hier_normal", S + 3, prior, x=y)
    ref = np.array([O.loglike(m, t) for t in th])
    pref = np.array([O.prior_loglike(m, t) for t in th])
    assert np.max(np.abs(ll - ref) / np.abs(ref)) <= RTOL
    assert np.max(np.abs(pr - pref) / np.abs(pref)) <= RTOL


# ---- (b) native RNG: posterior statistics -------------------------------------------------------
def test_native_binomial_posterior():
    """test/binomial_tests.jl restated: posterior is Beta(k+1, N-k+1)."""
    from scipy import stats
    rng = np.random.default_rng(29542)
    model = D.DEModel(sample_prior=lambda: [rng.uniform()], prior_loglike=D.GPUPrior(D.Beta(1, 1)),
                      loglike=D.GPULoglike("binomial", N=10, k=4), names=("θ",))
    de = D.DE(sample_prior=model.sample_prior, bounds=((0, 1),), burnin=1500, Np=3, seed=7)
    chains = D.sample(model, de, 3000)
    sol = stats.beta(5, 7)
    assert np.isclose(chains.mean()[0], sol.mean(), rtol=0.03)
    assert np.isclose(chains.std()[0], sol.std(), rtol=0.05)
    x = chains.value[::5, 0, :].ravel()
    assert stats.kstest(x, sol.cdf).statistic < 0.05   # the oracle's own chains give 0.01-0.03 here


def test_native_mvn_posterior_matches_oracle_chains():
    """Means, variances and KS statistics of the GPU chains against the oracle's chains (native RNG,
    different seeds) and against the analytic posterior sd = sigma/sqrt(n)."""
    from scipy import stats
    rng = np.random.default_rng(505514)
    n, dm, G, Np, n_iter, burn = 100, 8, 4, 16, 3000, 1000
    x = rng.normal(0.0, 1.0, size=(n, dm))
    case = common.Case("mvn", "mvnormal", dm + 1, [("normal", 0, 1)] * dm + [("halfcauchy", 0, 1)], [-np.inf] * dm + [0],
                       [np.inf] * (dm + 1), lambda r: list(r.normal(size=dm)) + [abs(r.standard_cauchy()) + 0.5], dict(x=x))
    theta0 = case.theta0(rng, G * Np)
    kw = dict(burnin=burn, theta_snooker=0.1)
    ref = O.run(case.oracle_config(G, Np, seed=11, **kw), case.oracle_model(), theta0, n_iter, record=False, trace=False)
    with case.handle(G, Np, seed=12, **kw) as h:
        h.set_state(theta0)
        h.run(n_iter)
        s = h.samples()
    a, b = s[:, :, burn:], ref["samples"][:, :, burn:]
    assert np.allclose(a.mean(axis=(0, 2)), b.mean(axis=(0, 2)), atol=0.02)
    assert np.allclose(a.std(axis=(0, 2)), b.std(axis=(0, 2)), rtol=0.08)
    assert np.allclose(a[:, :dm].std(axis=(0, 2)), 0.1, atol=0.02)
    assert np.corrcoef(a[:, :dm].mean(axis=(0, 2)), x.mean(axis=0))[0, 1] > 0.98
    for k in range(dm + 1):
        ks = stats.ks_2samp(a[:, k, ::20].ravel(), b[:, k, ::20].ravel()).statistic
        assert ks < 0.06, (k, ks)


def test_device_bundle_matches_bundle_samples():
    """demcmc_get_chains on the device = bundle_samples (main.jl:222-250), by-position quirk included."""
    from demcmc_b200.api import DE, DEModel, GPULoglike, GPUPrior, HalfCauchy, Normal, bundle_samples
    case = make_case("mvnormal", np.random.default_rng(23))
    G, Np = 3, 40
    theta0 = case.theta0(np.random.default_rng(5), G * Np)
    h = case.handle(G, Np, seed=5, burnin=10, alpha=0.6, theta_snooker=0.1)
    h.set_state(theta0)
    h.run(30)
    ids = h.get_state()[2]
    assert not np.array_equal(ids, np.arange(G * Np))
    d = theta0.shape[1]
    model = DEModel(sample_prior=lambda: [np.zeros(d - 1), 1.0], prior_loglike=GPUPrior(Normal(), HalfCauchy()),
                    loglike=GPULoglike("mvnormal", np.zeros((3, d - 1))), names=("mu", "sigma"))
    de = DE(sample_prior=model.sample_prior, bounds=((-1, 1), (0, 1)), n_groups=G, Np=Np, burnin=10)
    ref = bundle_samples(model, de, h.samples(), h.accept(), h.lp(), ids, [(d - 1,), ()], 30)
    assert np.array_equal(h.chains(10, 20).transpose(2, 1, 0), ref.value)
    h.close()


@pytest.mark.parametrize("mode", ["replay", "native"])
def test_blocking_on_as_a_function_of_the_iteration(mode):
    """blocking_on(de) is evaluated every iteration (main.jl:137,162): a schedule that switches block updating
    on and off -- block_update! over the blocks in some iterations, update! with all parameters in the others,
    consecutive unblocked iterations overlapped in one chunk."""
    case = make_case("hier_normal", np.random.default_rng(91))
    sched = [1, 0, 0, 0, 1, 1, 0, 0, 1, 0, 0, 0, 0, 1]
    r, out = forced_run(case, 2, 8, len(sched), mode, burnin=6, blocks=hier_blocks(9), alpha=0.3, blocking_schedule=sched)
    check(r, out)
    # unforced, as one call: same chain as iteration by iteration in native mode
    if mode == "native":
        theta0 = case.theta0(np.random.default_rng(0), 16)
        h = case.handle(2, 8, seed=5, burnin=6, blocks=hier_blocks(9), alpha=0.3, blocking_schedule=sched)
        h.set_state(theta0)
        h.run(len(sched))
        assert h.counters()["sweeps"] == sum(2 if s else 1 for s in sched)
        h.close()
    # unforced and short: runs of unblocked iterations share a chunk (overlapped sweeps with the blocks' sweep stride)
    sched2 = [0, 0, 0, 1, 0, 0, 0, 0]
    r, out = compare_run(case, 2, 8, len(sched2), mode, burnin=3, blocks=hier_blocks(9), alpha=0.3, blocking_schedule=sched2)
    assert np.array_equal(out["accept"], r["accept"])
    assert rel_err(out["samples"], r["samples"]) < 1e-9


def test_checkpoint_resume_is_exact():
    """run(a) + get_state + a NEW handle (set_state, set_weights, set_iteration) + run(b) = run(a + b): the
    Philox counters, the burn-in switch and the migration schedule continue (SURVEY 8f-4)."""
    for model, kw in (("mvnormal", dict(theta_snooker=0.2, alpha=0.3, burnin=14)), ("gaussian", dict(alpha=0.4, burnin=3, kappa=0.9))):
        case = make_case(model, np.random.default_rng(83))
        G, Np, a, b = 3, 8, 9, 11
        theta0 = case.theta0(np.random.default_rng(4), G * Np)
        h = case.handle(G, Np, seed=21, **kw)
        h.set_state(theta0)
        h.run(a + b)
        full = (h.history_by_slot(a, b), h.get_state())
        h.close()
        h1 = case.handle(G, Np, seed=21, **kw)
        h1.set_state(theta0)
        h1.run(a)
        th, w, ids = h1.get_state()
        h1.close()
        h2 = case.handle(G, Np, seed=21, **kw)
        h2.set_state(th, ids)
        h2.set_weights(w)
        h2.set_iteration(a)
        h2.run(b)
        res = (h2.history_by_slot(0, b), h2.get_state())
        h2.close()
        for x, y in zip(full[0] + full[1], res[0] + res[1]):
            assert np.array_equal(x, y)


def test_device_moments_match_the_chains():
    """demcmc_get_moments (k_moments_partial / k_moments_merge): pooled mean and variance per parameter of
    a row range of the history, against numpy on the downloaded rows; more vectors than blocks, fewer
    vectors than blocks, and d above one block of threads."""
    for model, kwm, G, Np, n_iter, row0 in (("mvnormal", {}, 4, 40, 30, 8), ("gaussian", {}, 2, 6, 12, 0),
                                            ("hier_normal", dict(n_obs=10, n_subjects=200), 2, 8, 6, 1)):
        case = make_case(model, np.random.default_rng(31), **kwm)
        h = case.handle(G, Np, seed=6, burnin=3, alpha=0.4)
        h.set_state(case.theta0(np.random.default_rng(8), G * Np))
        h.run(n_iter)
        th = h.history_by_slot(row0, n_iter - row0)[0]
        cnt, mean, var = h.moments(row0, n_iter - row0)
        flat = th.reshape(-1, th.shape[2])
        assert cnt == flat.shape[0]
        assert np.allclose(mean, flat.mean(axis=0), rtol=1e-12, atol=1e-13)
        assert np.allclose(var, flat.var(axis=0, ddof=1), rtol=1e-9, atol=1e-13)
        h.close()


# ---- de.sample = resample (DE-MCz, crossover.jl:113-124) and n_initial ---------------------------
@pytest.mark.parametrize("mode", ["replay", "native"])
@pytest.mark.parametrize("model", ["gaussian", "mvnormal", "lba"])
def test_resample_from_history(mode, model):
    case = make_case(model, np.random.default_rng(31))
    r, out = forced_run(case, 3, 6, 12, mode, burnin=6, n_initial=5, resample=True, theta_snooker=0.3, alpha=0.4)
    check(r, out, rtol_w=RTOL_W.get(model))
    assert np.array_equal(out["samples"][:, :, :5], r["samples"][:, :, :5])


@pytest.mark.parametrize("mode", ["replay", "native"])
def test_resample_blocking_hierarchical(mode):      # Examples/Hierarchical_Example.jl: blocks + resample + n_initial
    case = make_case("hier_normal", np.random.default_rng(32))
    r, out = forced_run(case, 2, 8, 10, mode, burnin=5, n_initial=4, resample=True, blocks=hier_blocks(9), alpha=0.3)
    check(r, out)


def test_sample_api_lnr_posterior():                 # test/lognormal_race_tests.jl at its own size
    common.lnr_posterior_check()


def test_sample_api_blocking_posterior():            # test/blocking_tests.jl at its own size
    common.blocking_posterior_check()


def test_sample_api_mvn_resample():                 # test/multivariate_normal_tests.jl at its own size
    common.mvn_resample_check(n_iter=50_000, burnin=5000, sd_atol=0.01)


def test_lanes_and_chunks_do_not_change_the_result():
    """Concurrent kernel chains over independent sets of groups (demcmc_set_lanes), programmatic
    dependent launch and overlapped chunks are execution schedules only: bit-identical chains."""
    case = make_case("mvnormal", np.random.default_rng(41), n_obs=3000)
    G, Np = 4, 48
    theta0 = case.theta0(np.random.default_rng(6), G * Np)
    outs = []
    for lanes, chunk in ((1, 1), (1, 16), (2, 16), (2, 3)):
        h = case.handle(G, Np, seed=8, burnin=6, theta_snooker=0.2, alpha=0.3)
        h.set_lanes(lanes)
        h.set_max_chunk(chunk)
        h.set_state(theta0)
        h.run(30)
        outs.append((h.samples(), h.accept(), h.lp(), h.get_state()[2]))
        h.close()
    for o in outs[1:]:
        assert all(np.array_equal(a, b) for a, b in zip(outs[0], o))


@pytest.mark.parametrize("model,kw", [("mvnormal", dict(theta_snooker=0.2, alpha=0.3, burnin=6)),
                                      ("mvnormal", dict(theta_snooker=0.0, alpha=0.1, burnin=0, kappa=0.8)),
                                      ("hier_normal", dict(theta_snooker=0.0, alpha=0.2, burnin=4))])
def test_persistent_chunk_kernel_is_a_schedule_only(model, kw, monkeypatch):
    """k_chunk_persist (all levels of a chunk in one warp-specialised launch: DMMA warps, helper warps,
    scalar CTAs, counter-based dependencies, two alternating lanes) against the level-by-level
    launches of k_propose / k_xdot / k_accept: bit-identical chains, and the counters show which
    path ran."""
    case = make_case(model, np.random.default_rng(43), n_obs=4000 if model == "mvnormal" else 700)
    if model == "hier_normal":
        kw = dict(kw, blocks=hier_blocks(case.d - 3))          # blocking_on: every block is its own chunk
    G, Np = 4, 40
    theta0 = case.theta0(np.random.default_rng(7), G * Np)
    outs, chunks, launches = [], [], []
    for persist in ("0", "1"):
        monkeypatch.setenv("DEMCMC_PERSIST", persist)
        h = case.handle(G, Np, seed=9, **kw)
        h.set_state(theta0)
        h.run(40)
        c = h.counters()
        outs.append((h.samples(), h.accept(), h.lp(), h.get_state()[2]))
        chunks.append(c["persistent_chunks"]); launches.append(c["kernel_launches"])
        h.close()
    assert chunks[0] == 0 and chunks[1] > 0, chunks
    assert launches[1] < launches[0] / 4, launches
    assert all(np.array_equal(a, b) for a, b in zip(outs[0], outs[1]))


def test_persistent_chunk_kernel_replays_the_oracle(monkeypatch):
    """Replay through the persistent kernel: the reference's draws from the tape, accept decisions
    identical to the oracle's, log densities within 1e-12 relative (teacher-forced per iteration)."""
    monkeypatch.setenv("DEMCMC_PERSIST", "1")
    case = make_case("mvnormal", np.random.default_rng(47), n_obs=2500)
    r, out = forced_run(case, 4, 24, 12, "replay", burnin=5, theta_snooker=0.15, alpha=0.3)
    check(r, out)


@pytest.mark.parametrize("mode", ["replay", "native"])
def test_wide_kernels_long_parameter_vectors(mode, monkeypatch):
    """d >= 256 (hierarchical normal with 300 subjects, d = 303, parameter blocks): the proposal and the
    accept run as one CTA of 256 threads per particle (k_propose_wide / k_accept_wide) -- same
    accept decisions as the oracle, values within 1e-12; and the same chain as the one-warp kernels."""
    monkeypatch.setenv("DEMCMC_PERSIST", "0")                 # (a population this small would otherwise run in the persistent kernel)
    case = make_case("hier_normal", np.random.default_rng(61), n_obs=20, n_subjects=300)
    S = case.d - 3
    r, out = forced_run(case, 2, 10, 8, mode, burnin=4, blocks=hier_blocks(S), alpha=0.3)
    check(r, out)
    theta0 = case.theta0(np.random.default_rng(3), 2 * 10)
    outs = []
    for no_wide in ("1", "0"):
        monkeypatch.setenv("DEMCMC_NO_WIDE", no_wide)
        h = case.handle(2, 10, seed=4, burnin=3, blocks=hier_blocks(S), alpha=0.3)
        h.set_state(theta0)
        h.run(12)
        assert h.counters()["persistent_chunks"] == 0
        outs.append((h.samples(), h.accept(), h.lp()))
        h.close()
    assert np.array_equal(outs[0][1], outs[1][1])                       # accept decisions
    assert np.allclose(outs[0][0], outs[1][0], rtol=1e-9, atol=1e-12)    # reductions differ in order only
    fin = np.isfinite(outs[0][2])
    assert np.allclose(outs[0][2][fin], outs[1][2][fin], rtol=1e-9, atol=1e-9)


@pytest.mark.parametrize("mode", ["replay", "native"])
@pytest.mark.parametrize("model,kw", [
    ("hier_normal", dict(blocks=True, theta_snooker=0.2, alpha=0.3)),            # blocks + snooker + the NORMAL_REF prior
    ("hier_normal", dict(theta_snooker=0.15, kappa=0.7, burnin=6)),              # recombination + the burn-in base term
    ("mvnormal", dict(theta_snooker=0.1, alpha=0.3, kappa=0.9)),                 # d = 301: the means staged from registers
    ("hier_normal", dict(resample=True, n_initial=4, theta_snooker=0.2)),        # DE-MCz: donors are cells of the history
])
def test_one_pass_wide_proposal(mode, model, kw, monkeypatch):
    """k_propose_wide1 (four elements per thread, one pass, d <= 1024): the oracle's accept decisions and values, and
    the chain of the three-pass kernel k_propose_wide (same per-element arithmetic, other summation order for the mean
    square only)."""
    kw = dict(kw)
    rng = np.random.default_rng(67)
    if model == "hier_normal":
        case = make_case("hier_normal", rng, n_obs=12, n_subjects=297)           # d = 300: last pair of elements incomplete
        if kw.pop("blocks", False):
            kw["blocks"] = hier_blocks(case.d - 3)
    else:
        case = make_case("mvnormal", rng, n_obs=300, n_dim=300)
    kw.setdefault("burnin", 4)
    monkeypatch.setenv("DEMCMC_PERSIST", "0")                 # the level-by-level path: that is where the wide kernels are
    monkeypatch.setenv("DEMCMC_WIDE_SHAPE", "5")
    r, out = forced_run(case, 2, 9, 8, mode, **kw)
    check(r, out)
    theta0 = case.theta0(np.random.default_rng(3), 2 * 9)
    rows = np.stack([case.theta0(np.random.default_rng(40 + i), 2 * 9) for i in range(kw["n_initial"])]) if kw.get("resample") else None
    outs, names = [], []
    for shape in ("0", "32", "35"):
        monkeypatch.setenv("DEMCMC_WIDE_SHAPE", shape)
        h = case.handle(2, 9, seed=4, **kw)
        if rows is not None:
            h.set_history(rows)
            h.set_state(None)
        else:
            h.set_state(theta0)
        h.run(12)
        assert h.counters()["persistent_chunks"] == 0
        outs.append((h.samples(), h.accept(), h.lp()))
        h.close()
    for other in outs[1:]:
        assert np.array_equal(outs[0][1], other[1])
        assert np.allclose(outs[0][0], other[0], rtol=1e-9, atol=1e-12)
        fin = np.isfinite(outs[0][2])
        assert np.allclose(outs[0][2][fin], other[2][fin], rtol=1e-9, atol=1e-9)


@pytest.mark.parametrize("mode", ["replay", "native"])
def test_one_pass_wide_proposal_at_the_configs3_length(mode, monkeypatch):
    """d = 1003 (1000 subjects, two parameter blocks): all four elements of every thread in use, the last trip partial;
    20 dimension splits of the short-stream k_xdot; two lanes.  Oracle parity, teacher-forced."""
    monkeypatch.setenv("DEMCMC_PERSIST", "0")
    case = make_case("hier_normal", np.random.default_rng(83), n_obs=50, n_subjects=1000)
    r, out = forced_run(case, 2, 7, 5, mode, burnin=2, blocks=hier_blocks(1000), theta_snooker=0.2, alpha=0.3)
    check(r, out)


# ---- the optimize path (optimize.jl; maximize! / minimize! + evaluate_fun!) -------------------------
@pytest.mark.parametrize("mode", ["replay", "native"])
@pytest.mark.parametrize("model,update", [("rastrigin", "minimize"), ("gaussian", "maximize"), ("mvnormal", "maximize")])
def test_optimize_updates(mode, model, update):
    case = make_case(model, np.random.default_rng(51))
    r, out = forced_run(case, 2, 6, 25, mode, burnin=10, update=update, fitness="fun", alpha=0.3)
    check(r, out)
    assert not out["accept"].any() and not out["lp"].any()


def test_optimize_api():                            # test/optimization_tests.jl at its own size
    common.optimize_checks()


# ---- thinning and the multi-device handle: the bodies of the CPU tests, on the device ---------------------------------
import test_host_logic_emu as E  # noqa: E402


@pytest.mark.parametrize("model,kw", [("mvnormal", dict(theta_snooker=0.2, alpha=0.4)), ("gaussian", dict(kappa=0.8)),
                                      ("hier_normal", dict(blocks=True, alpha=0.3))])
def test_thinned_run_keeps_every_kth_row_of_the_full_run(model, kw):
    E.test_thinned_run_keeps_every_kth_row_of_the_full_run(None, model, kw)


def test_thinned_resample_runs_on_the_stored_rows():
    E.test_thinned_resample_runs_on_the_stored_rows(None)


@pytest.mark.parametrize("model,kw", [("mvnormal", dict(theta_snooker=0.25, alpha=0.4, burnin=6)), ("gaussian", dict(kappa=0.8)),
                                      ("mvnormal", dict(resample=True, theta_snooker=0.2, burnin=3))])
def test_plan_records_equal_the_draws_made_in_place(model, kw, monkeypatch):
    E.test_plan_records_equal_the_draws_made_in_place(None, model, kw, monkeypatch)


def test_thinned_run_through_the_persistent_kernel():
    """configs[1]-like shape: chunks of 16 overlapped sweeps write 15 scratch rows + 1 history row each"""
    rng = np.random.default_rng(6)
    case = make_case("mvnormal", rng, n_obs=3000)
    G, Np, n_iter = 4, 64, 48
    th0 = case.theta0(rng, G * Np)
    outs = []
    for every in (1, 16, 5):
        with case.handle(G, Np, seed=3, burnin=5, alpha=0.05, theta_snooker=0.1, store_every=every) as h:
            h.set_state(th0)
            h.run(n_iter)
            outs.append((h.samples(), h.get_state(), h.counters()))
    assert outs[0][2]["persistent_chunks"] > 0 and outs[1][2]["persistent_chunks"] > 0
    assert np.array_equal(outs[1][0], outs[0][0][:, :, 15::16]) and np.array_equal(outs[2][0], outs[0][0][:, :, 4::5])
    assert all(np.array_equal(a, b) for a, b in zip(outs[1][1], outs[0][1]))


def _n_gpus():
    return D._ffi.lib().demcmc_device_count()


@pytest.mark.parametrize("model,kw", [("mvnormal", dict(theta_snooker=0.2, alpha=0.6)), ("lnr", dict(alpha=0.5)),
                                      ("hier_normal", dict(blocks=True, alpha=0.5, store_every=2)),
                                      ("mvnormal", dict(resample=True, n_initial=5, theta_snooker=0.2, alpha=0.6)),
                                      ("hier_normal", dict(blocks=True, resample=True, n_initial=4, alpha=0.5))])
def test_multi_device_handle_is_the_single_device_chain(model, kw):
    if _n_gpus() < 2:
        pytest.skip("a multi-device handle needs two GPUs (gpurun --gpus 2)")
    E.test_multi_device_handle_is_the_single_device_chain(None, model, kw, 2)
    if _n_gpus() >= 4:
        E.test_multi_device_handle_is_the_single_device_chain(None, model, kw, 4)


def test_multi_device_handle_replays_the_oracle():
    if _n_gpus() < 2:
        pytest.skip("a multi-device handle needs two GPUs (gpurun --gpus 2)")
    E.test_multi_device_handle_replays_the_oracle_and_checks_its_arguments(None)


def test_multi_device_sample_api_at_configs1_shape():
    """sample(model, de, n_iter, devices=[...]) from ONE process: the single-GPU chains bit for bit (persistent kernel on
    every device, migration through the peer-mapped mailboxes)"""
    if _n_gpus() < 2:
        pytest.skip("a multi-device handle needs two GPUs (gpurun --gpus 2)")
    rng = np.random.default_rng(50514)
    n, dm, G, Np, n_iter = 20_000, 50, 8, 64, 60
    x = rng.normal(rng.normal(size=dm), 1.0, size=(n, dm))
    outs = []
    for devices in (None, list(range(min(_n_gpus(), 4)))):
        r2 = np.random.default_rng(1)
        model = D.DEModel(sample_prior=lambda: [r2.normal(size=dm), abs(r2.standard_cauchy()) + 0.2], prior_loglike=D.GPUPrior(D.Normal(0, 1), D.HalfCauchy(0, 1)),
                          loglike=D.GPULoglike("mvnormal", x), names=("μ", "σ"))
        de = D.DE(sample_prior=model.sample_prior, bounds=((-np.inf, np.inf), (0.0, np.inf)), n_groups=G, Np=Np, burnin=10, θsnooker=0.1, α=0.3, seed=5)
        outs.append(D.sample(model, de, n_iter, devices=devices).value)
    assert np.array_equal(outs[0], outs[1])


def test_device_diagnostics_match_the_host_estimators():
    E._check_device_diagnostics()
    E._check_device_diagnostics(n_iter=91)
    E._check_device_diagnostics(store_every=2, n_iter=120)
    E._check_device_diagnostics(G=4, Np=64, n_iter=400)
    if _n_gpus() >= 2:
        E._check_device_diagnostics(devices=[0, 1])


def test_device_diagnostics_of_long_chains(monkeypatch):
    """more than 8192 stored rows (the split chain in opted-in shared memory), and the lags in several batches
    (k_diag_partial with lag0 > 0) against the one-batch result and the host estimators"""
    E._check_device_diagnostics(G=2, Np=4, n_iter=12000)
    monkeypatch.setenv("DEMCMC_DIAG_LAGS", "8")
    E._check_device_diagnostics(G=2, Np=5, n_iter=300)
    monkeypatch.setenv("DEMCMC_DIAG_LAGS", "512")
    E._check_device_diagnostics(G=2, Np=4, n_iter=12000)


def test_full_covariance_mvn_kernel():          # SURVEY 8f-4
    E._check_mvn_full()
    # a larger, strongly correlated case through the persistent kernel against the oracle's per-observation whitening
    rng = np.random.default_rng(17)
    n, dm = 4000, 50
    A = rng.normal(size=(dm, dm))
    cov = A @ A.T / dm + 0.2 * np.eye(dm)
    mu = rng.normal(size=dm)
    x = rng.multivariate_normal(mu, cov, size=n)
    prior = [("normal", 0, 2)] * dm + [("halfcauchy", 0, 1)]
    case = common.Case("mvn_full50", "mvnormal_full", dm + 1, prior, [-np.inf] * dm + [0], [np.inf] * (dm + 1),
                       lambda r: list(r.normal(mu, 0.05)) + [abs(r.normal(1, 0.05))], dict(x=x, cov=cov))
    r, out = forced_run(case, 4, 16, 3, "replay", burnin=1, theta_snooker=0.1)
    assert out["counters"]["persistent_chunks"] > 0
    check(r, out)
    # data 1e4 sd from 0 under a covariance of condition 1e6: the oracle whitens x_i - mu per observation, which does
    # not cancel at the offset; the library centres before whitening for the same reason.  Crossover moves only: the
    # snooker projection (utilities.jl:239-246) takes dot products of the UNCENTRED donor with a difference of size
    # the spread, so at this offset the warp-order sums of the device and the oracle's sequential ones give proposals
    # that differ by more than 1e-12 before any likelihood is evaluated (the snooker path is covered above)
    dm = 10
    q, _ = np.linalg.qr(rng.normal(size=(dm, dm)))
    cov = (q * np.geomspace(1.0, 1e-6, dm)) @ q.T
    cov = (cov + cov.T) / 2.0
    mu = 1e4 * (1.0 + rng.uniform(size=dm))
    x = rng.multivariate_normal(mu, cov, size=n)
    xbar = x.mean(axis=0)
    case = common.Case("mvn_full_offset", "mvnormal_full", dm + 1, [("flat",)] * dm + [("halfcauchy", 0, 1)],
                       [-np.inf] * dm + [0], [np.inf] * (dm + 1),
                       lambda r: list(rng.multivariate_normal(xbar, cov / n)) + [abs(r.normal(1, 0.05))], dict(x=x, cov=cov))
    r, out = forced_run(case, 4, 16, 3, "replay", burnin=1, theta_snooker=0.0)
    assert out["counters"]["persistent_chunks"] > 0
    check(r, out)


def test_vector_parameter_gaussian_example():   # Examples/Guassian_Example_Vector.jl
    E._check_vector_gaussian_example()


@pytest.mark.parametrize("kw", [dict(alpha=0.3), dict(alpha=0.0, proposal="fixed_gamma", kappa=0.8), dict(alpha=0.2, store_every=3)])
def test_overlapped_block_sweeps_are_a_schedule_only(kw):
    E.test_overlapped_block_sweeps_are_a_schedule_only(None, kw)


def test_overlapped_block_sweeps_wide_kernels(monkeypatch):
    """the configs[3] shape in small: 300 subjects (d = 303: the one-CTA-per-particle kernels), two blocks"""
    monkeypatch.setenv("DEMCMC_PERSIST", "0")
    rng = np.random.default_rng(2)
    case = make_case("hier_normal", rng, n_subjects=300)
    th0 = case.theta0(rng, 4 * 24)
    outs = []
    for chunk in (1, 16):
        with case.handle(4, 24, seed=6, burnin=0, blocks=hier_blocks(300), alpha=0.2) as h:
            h.set_max_chunk(chunk)
            h.set_state(th0)
            h.run(12)
            outs.append((h.samples(), h.accept(), h.counters()["levels"]))
    assert np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][1], outs[1][1]) and outs[1][2] < outs[0][2]

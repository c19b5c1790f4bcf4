"""The summaries of the stored history that a user reads instead of downloading the draws: split-R-hat and ESS
(demcmc_get_diagnostics: k_diag_partial / k_diag_merge, then diag_finish) and the pooled moments (demcmc_get_moments:
k_moments_partial / k_moments_merge, Chan's merge across the devices of a multi-device handle).

Every check runs on the host-only test double and, with -m gpu, on the CUDA backend.  The reference is written here in
np.longdouble from the definitions, independently of diagnostics.py (a float64 implementation, itself under test): two-pass
chain means and variances, direct lag sums for the autocovariances, Geyer's initial positive, monotone pair sequence.
Most inputs are injected as prior rows (n_initial = N, resample = True, set_history), so the rows are exactly the ones the
test chose; the rest come from real runs.  The inputs include parameters at large offsets with a small spread (intercepts,
scales, times), where one-pass sums of uncentred draws lose the between-chain variance."""
import math
from fractions import Fraction

import numpy as np
import pytest

import common
from common import D, make_case

LD = np.longdouble
EUNSUPPORTED = -6

# Tolerances: 100x the larger of the worst errors measured over every case of this file on the test double and on one
# B200 (1000 W power limit; the two-device cases ran on the test double only).  R-hat: absolute; ESS: relative; mean:
# relative to max(|mean|, sd); variance: relative.  Measured: test double / B200.
TOL_RHAT = 2e-11     # 2.0e-13 / 2.0e-13 (66 chains of 20 draws, d = 129, offsets up to 1e8 sd)
TOL_ESS = 4e-10      # 4.7e-12 / 4.7e-12 (the same case)
TOL_MEAN = 5e-13     # 5.5e-15 / 2.8e-15
TOL_VAR = 7e-10      # 7.7e-12 / 2.4e-15 (test double: two devices at 1e8 sd, Chan's merge of the two shards' means)
GEYER_MARGIN = 1e-6  # a reference pair sum this close to 0 could flip the truncation through rounding: choose other inputs


@pytest.fixture(params=["emu", pytest.param("cuda", marks=pytest.mark.gpu)])
def backend(request):
    """Binds the test double or the CUDA library for one test (the conftest fixtures set each up once per session)."""
    request.getfixturevalue(request.param)
    if request.param == "cuda":
        common.use_cuda()
    else:
        D._ffi.use_library(common.EMU_LIB)
    return request.param


def _n_devices():
    return D._ffi.lib().demcmc_device_count()


# ---- the reference -----------------------------------------------------------------------------------------------------
def _halves(chains):
    """chains [m][n_rows] -> the 2m split chains [2m][nh] in longdouble: nh = n_rows // 2, the middle draw dropped when
    n_rows is odd (backend.h: launch_diag_aggregates)"""
    x = np.asarray(chains, dtype=LD)
    n_rows = x.shape[1]
    nh = n_rows // 2
    return np.concatenate([x[:, :nh], x[:, n_rows - nh:]])


def _exact(v):
    return Fraction(*LD(v).as_integer_ratio())


def ref_diagnostics(chains):
    """(split-R-hat, ESS, margin, stop lag) of one parameter, chains [m][n_rows] (float64 draws); R-hat and ESS in
    longdouble.  margin = the smallest
    |pair sum| Geyer's sequence evaluated, the stopping pair included; stop lag = the even lag t of the pair that ended it
    (nh when none did)."""
    x = _halves(chains)
    M, nh = x.shape
    means = x.sum(axis=1) / nh
    xc = x - means[:, None]
    W = (xc * xc).sum() / (nh - 1) / M
    gm = means.sum() / M
    var_means = ((means - gm) ** 2).sum() / (M - 1)
    var_plus = W * (nh - 1) / nh + var_means
    rhat = np.sqrt(var_plus / W) if W > 0 else LD(math.nan)
    if not var_plus > 0:
        return rhat, LD(math.nan), math.inf, 0

    def rho(t):          # biased autocovariance at lag t summed over the chains, direct sum
        return LD(1) if t == 0 else 1 - (W - (xc[:, :nh - t] * xc[:, t:]).sum() / nh / M) / var_plus
    tau, prev, margin, t = LD(-1), LD(math.inf), math.inf, 0
    while t + 1 < nh:
        pair = rho(t) + rho(t + 1)
        margin = min(margin, abs(float(pair)))
        if pair < 0:
            break
        pair = min(pair, prev)
        prev = pair
        tau += 2 * pair
        t += 2
    tau = max(tau, 1 / LD(math.log10(max(nh * M, 10))))
    return rhat, nh * M / tau, margin, t


def ref_moments(draws):
    """two-pass mean and variance (ddof 1) of all draws, in longdouble"""
    x = np.asarray(draws, dtype=LD).reshape(-1)
    m = x.sum() / x.size
    return float(m), float(((x - m) ** 2).sum() / (x.size - 1))


# ---- comparisons -------------------------------------------------------------------------------------------------------
WORST = {"rhat": 0.0, "ess": 0.0, "mean": 0.0, "var": 0.0}    # largest errors seen in this session (for the tolerances)


def _note(kind, err):
    WORST[kind] = max(WORST[kind], err)
    return err


def check_diagnostics(h, row0, n, what=""):
    """h.diagnostics(row0, n) against the reference on the chains by id from samples()"""
    rhat, ess = h.diagnostics(row0, n)
    s = h.samples()[:, :, row0:row0 + n]
    bad = []
    for k in range(h.d):
        r_rhat, r_ess, margin, _ = ref_diagnostics(s[:, k, :])
        r_rhat, r_ess = float(r_rhat), float(r_ess)
        assert margin > GEYER_MARGIN, (what, k, margin)
        if math.isnan(r_rhat) or math.isnan(r_ess):
            if not (np.isnan(rhat[k]) == math.isnan(r_rhat) and np.isnan(ess[k]) == math.isnan(r_ess)):
                bad.append((k, "NaN pattern", rhat[k], r_rhat, ess[k], r_ess))
            continue
        e_r = _note("rhat", abs(rhat[k] - r_rhat))
        e_e = _note("ess", abs(ess[k] - r_ess) / r_ess)
        if not (e_r <= TOL_RHAT and e_e <= TOL_ESS):
            bad.append((k, f"|dRhat| {e_r:.3g} rel dESS {e_e:.3g}", float(rhat[k]), r_rhat, float(ess[k]), r_ess))
    assert not bad, (what, bad)


def check_moments(h, row0, n, what=""):
    """h.moments(row0, n) against the reference over every particle's draws of those rows"""
    cnt, mean, var = h.moments(row0, n)
    s = h.samples()[:, :, row0:row0 + n]
    assert cnt == s.shape[0] * s.shape[2], (what, cnt)
    bad = []
    for k in range(h.d):
        r_mean, r_var = ref_moments(s[:, k, :])
        e_m = _note("mean", abs(mean[k] - r_mean) / max(abs(r_mean), math.sqrt(r_var)) if r_var > 0 else abs(mean[k] - r_mean))
        e_v = _note("var", abs(var[k] - r_var) / r_var if r_var > 0 else abs(var[k]))
        if not ((e_m <= TOL_MEAN or (r_var == 0 and mean[k] == r_mean)) and (e_v <= TOL_VAR or (r_var == 0 and var[k] == 0))):
            bad.append((k, f"mean err {e_m:.3g} var err {e_v:.3g}", float(mean[k]), r_mean, float(var[k]), r_var))
    assert not bad, (what, bad)


def injected(rows, G, Np, devices=None):
    """A handle whose history is exactly rows [N][P][d] (row i, slot p = particle id p), with no run"""
    N, P, d = rows.shape
    assert P == G * Np
    h = D.Handle(G, Np, d, np.full(d, -np.inf), np.full(d, np.inf), n_initial=N, resample=True, devices=devices)
    h.set_history(rows)
    assert np.array_equal(h.samples(), np.transpose(rows, (1, 2, 0)))
    return h


def check_injected(rows, G, Np, what="", devices=None, moments=True):
    N = rows.shape[0]
    with injected(rows, G, Np, devices) as h:
        check_diagnostics(h, 0, N, what)
        if moments:
            check_moments(h, 0, N, what)


def iid_rows(rng, N, P, offsets, sds, chain_shift=0.05):
    """N(offset_k + chain_shift * sd_k * u_id, sd_k) draws: i.i.d. within a chain, the chains a little apart"""
    offsets, sds = np.asarray(offsets, float), np.asarray(sds, float)
    u = rng.normal(size=(1, P, offsets.size))
    return offsets + sds * (rng.normal(size=(N, P, offsets.size)) + chain_shift * u)


def ar1_rows(rng, N, P, phi, d=2):
    x = np.empty((N, P, d))
    x[0] = rng.normal(size=(P, d)) / math.sqrt(1 - phi * phi)
    for i in range(1, N):
        x[i] = phi * x[i - 1] + rng.normal(size=(P, d))
    return x


# ---- the reference against exact rational arithmetic -------------------------------------------------------------------
def test_reference_against_exact_arithmetic():
    """R-hat^2 and the first autocovariances of the longdouble reference against fractions.Fraction on the same float64
    draws (3 chains of 9 rows: the middle row is dropped, nh = 4, 6 split chains)"""
    assert np.finfo(LD).eps <= 2.0 ** -63, "the reference needs an extended-precision long double"
    rng = np.random.default_rng(41)
    chains = 1e3 + rng.normal(size=(3, 9)) * 0.01
    halves = [[Fraction(float(v)) for v in c[:4]] for c in chains] + [[Fraction(float(v)) for v in c[5:]] for c in chains]
    M, nh = len(halves), 4
    means = [sum(c) / nh for c in halves]
    W = sum(sum((v - m) ** 2 for v in c) / (nh - 1) for c, m in zip(halves, means)) / M
    gm = sum(means) / M
    var_plus = W * Fraction(nh - 1, nh) + sum((m - gm) ** 2 for m in means) / (M - 1)
    rhat2 = var_plus / W
    r_rhat = ref_diagnostics(chains)[0]
    assert abs(_exact(r_rhat) ** 2 - rhat2) <= Fraction(1, 10 ** 17) * rhat2, (float(r_rhat), float(rhat2))
    x = _halves(chains)
    xc = x - (x.sum(axis=1) / nh)[:, None]
    for t in range(4):
        exact = sum(sum((c[i] - m) * (c[i + t] - m) for i in range(nh - t)) for c, m in zip(halves, means)) / nh
        got = (xc[:, :nh - t] * xc[:, t:]).sum() / nh
        assert abs(_exact(got) - exact) <= Fraction(1, 10 ** 15) * W, (t, float(got), float(exact))


# ---- injected rows -----------------------------------------------------------------------------------------------------
RATIOS = np.array([0.0, 1e4, 1e6, 1e7, 1e8])


@pytest.mark.parametrize("N,G,Np,d,row0", [(1000, 2, 8, 6, 0), (600, 1, 3, 5, 0), (5, 1, 4, 5, 0), (40, 3, 11, 129, 0),
                                           (12291, 1, 3, 5, 0), (300, 2, 4, 5, 17)])
def test_large_offsets(backend, N, G, Np, d, row0):
    """offset / sd of 0, 1e4, 1e6, 1e7 and 1e8, different ones in different parameters of one handle, of either sign and
    with spreads from 1e-4 to 3: the between-chain variance of chain means near 1e8 sd must not cancel.  2 x 8 chains of
    1000 draws; 6 split chains; nh = 2; 66 chains and d = 129; nh = 6145 (opted-in shared memory); a range from row 17"""
    rng = np.random.default_rng(N + d)
    ratios = RATIOS[np.arange(d) % 5]
    sds = np.array([1.0, 3e-4, 2.5, 1e-2, 7e-5, 3.0])[np.arange(d) % 6]
    offsets = ratios * sds * np.where(np.arange(d) % 3 == 2, -1.0, 1.0)
    with injected(iid_rows(rng, N, G * Np, offsets, sds, chain_shift=0.3 if N < 100 else 0.05), G, Np) as h:
        check_diagnostics(h, row0, N - row0, "offsets")
        check_moments(h, row0, N - row0, "offsets")


def test_degenerate_parameters(backend):
    """a parameter constant in every chain (no spread: R-hat and ESS NaN, at any value), one chain constant while the
    others move, and heavy ties"""
    rng = np.random.default_rng(2)
    N, P = 200, 6
    rows = np.empty((N, P, 6))
    rows[:, :, 0] = 0.5                                               # constant everywhere, a sum of it is exact
    rows[:, :, 1] = 3.7e-3                                            # constant everywhere, a sum of it rounds
    rows[:, :, 2] = rng.normal(size=(N, P))
    rows[:, 0, 2] = 0.3                                               # the chain of id 0 constant
    rows[:, :, 3] = rng.normal(size=(N, P))
    rows[:, 3, 3] = -2.0                                              # another chain constant
    rows[:, :, 4] = rng.integers(0, 3, size=(N, P)) * 0.25            # three values only
    rows[:, :, 5] = rng.integers(0, 2, size=(N, P)) * 1e-3 + (np.arange(N) % 2)[:, None] * 1e-3
    with injected(rows, 1, P) as h:
        rhat, ess = h.diagnostics(0, N)
        assert np.isnan(rhat[:2]).all() and np.isnan(ess[:2]).all(), (rhat, ess)
        check_diagnostics(h, 0, N, "degenerate")
        check_moments(h, 0, N, "degenerate")
        assert (h.moments(0, N)[2][:2] == 0.0).all()


@pytest.mark.parametrize("phi", [0.9, 0.99])
@pytest.mark.parametrize("lags", [None, "2", "6"])
def test_autocorrelated_chains(backend, monkeypatch, phi, lags):
    """AR(1) chains: Geyer's sequence runs for tens to hundreds of lags, through many batches of lags when the batch is
    small"""
    if lags:
        monkeypatch.setenv("DEMCMC_DIAG_LAGS", lags)
    rng = np.random.default_rng(3 if phi == 0.9 else 4)
    rows = ar1_rows(rng, 1601, 5, phi)
    rows[:, :, 1] *= 0.01
    check_injected(rows, 1, 5, f"AR(1) phi {phi}", moments=lags is None)


def test_geyer_sequence_stopping_at_a_batch_boundary(backend, monkeypatch):
    """the sequence ends on the first pair of a batch of lags, on its last pair, and one pair after a batch"""
    rng = np.random.default_rng(5)
    rows = ar1_rows(rng, 400, 3, 0.8, d=1)
    stop = ref_diagnostics(rows[:, :, 0].T)[3]
    assert 4 <= stop < 100, stop
    for step in (stop, stop + 2, stop - 2):
        monkeypatch.setenv("DEMCMC_DIAG_LAGS", str(step))
        check_injected(rows, 1, 3, f"batches of {step} lags, stop at lag {stop}", moments=False)


@pytest.mark.parametrize("n_rows", [4, 5, 6, 7, 1000, 1001])
def test_short_and_odd_chains(backend, n_rows):
    """nh = 2 (4 and 5 rows), odd numbers of rows (the middle draw dropped)"""
    rng = np.random.default_rng(6 + n_rows)
    check_injected(iid_rows(rng, n_rows, 4, [0.0, 3.0], [1.0, 0.5], chain_shift=0.3), 1, 4, f"{n_rows} rows")


@pytest.mark.parametrize("nh", [6144, 6145, 24576])
def test_split_chain_in_shared_memory(backend, nh):
    """the longest split chain within the default 48 KB of shared memory, the first beyond it (opt-in), and the longest
    one call holds (DG_MAX_NH)"""
    rng = np.random.default_rng(nh)
    check_injected(iid_rows(rng, 2 * nh + (nh == 6145), 3, [0.0], [1.0]), 1, 3, f"nh {nh}")


def test_too_long_a_range_is_refused(backend):
    rows = np.random.default_rng(7).normal(size=(49154, 3, 1))
    with injected(rows, 1, 3) as h:
        with pytest.raises(D._ffi.DemcmcError) as e:
            h.diagnostics(0, 49154)
        assert e.value.code == EUNSUPPORTED


@pytest.mark.parametrize("G,Np", [(1, 3), (1, 5), (4, 4), (3, 11), (8, 6)])
def test_chain_counts(backend, G, Np):
    """6, 10, 32, 66 and 96 split chains: fewer than the 32 groups of chains k_diag_partial reduces, as many, more and not
    a multiple, a multiple (a handle holds at least 3 particles)"""
    rng = np.random.default_rng(100 + G * Np)
    check_injected(iid_rows(rng, 301, G * Np, [0.0, -0.6, 0.9], [1.0, 1e-1, 2.0], chain_shift=0.2), G, Np, f"{2 * G * Np} chains")


@pytest.mark.parametrize("d", [1, 129, 300])
def test_many_parameters(backend, d):
    """d above one block of moment threads (128): the loop over parameters wraps"""
    rng = np.random.default_rng(d)
    sds = np.exp(rng.uniform(-8, 3, size=d))
    check_injected(iid_rows(rng, 80, 5, rng.normal(size=d) * sds, sds, chain_shift=0.3), 1, 5, f"d {d}")


@pytest.mark.parametrize("N,G,Np", [(197, 1, 3), (148, 1, 4), (1, 1, 593), (395, 1, 3), (3, 4, 50)])
def test_moments_around_the_block_count(backend, N, G, Np):
    """N x P vectors of 591, 592 (the moment kernel's block count), 593 and 1185, and 600 with d = 130"""
    rng = np.random.default_rng(N * Np)
    d = 130 if G == 4 else 3
    rows = iid_rows(rng, N, G * Np, np.arange(d) % 3, np.full(d, 0.5))
    with injected(rows, G, Np) as h:
        check_moments(h, 0, N, f"{N * G * Np} vectors")
        if N >= 3:
            check_moments(h, 1, N - 2, "inner rows")


def test_injected_rows_on_two_devices(backend):
    """offset rows on a handle over two devices (two shards on the test double): one shift for every shard"""
    if backend == "cuda" and _n_devices() < 2:
        pytest.skip("needs two GPUs")
    rng = np.random.default_rng(8)
    sds = np.array([1.0, 0.01, 3.0])
    check_injected(iid_rows(rng, 500, 16, np.array([0.0, 1e6, 1e8]) * sds, sds), 4, 4, "two devices", devices=[0, 1])


# ---- rows of real runs -------------------------------------------------------------------------------------------------
def _gaussian(centre, n_obs=300):
    """the Gaussian model with flat priors on data centred at `centre` with sd 0.01: the posterior sd of mu is ~6e-4"""
    rng = np.random.default_rng(9)
    case = make_case("gaussian", rng, n_obs=n_obs)
    case.data = dict(x=centre + 0.01 * rng.normal(size=n_obs))
    case.prior = [("flat",), ("flat",)]
    case.sample_prior = lambda r: [centre + 0.001 * r.normal(), 0.01 * (1 + 0.1 * abs(r.normal()))]
    return case


@pytest.mark.parametrize("centre", [0.0, 1e4])
@pytest.mark.parametrize("devices", [None, [0, 1]])
def test_run_with_migrating_ids(backend, devices, centre):
    """alpha > 0: ids change slots (and devices); thinned rows (store_every = 3); the chains by id from samples()"""
    if devices and backend == "cuda" and _n_devices() < 2:
        pytest.skip("needs two GPUs")
    case = _gaussian(centre)
    G, Np = 4, 6
    with case.handle(G, Np, seed=3, burnin=0, alpha=0.4, store_every=3, devices=devices) as h:
        h.set_state(case.theta0(np.random.default_rng(1), G * Np))
        h.run(600)
        ids = h.history_by_slot()[2]
        assert (ids != ids[0]).any(), "no migration"
        check_diagnostics(h, 40, h.n_rows - 40, "migrating ids")
        check_moments(h, 40, h.n_rows - 40, "migrating ids")


def _run_after_prior_rows(centre):
    case = _gaussian(centre)
    G, Np, n0, n_iter = 3, 6, 40, 90
    rng = np.random.default_rng(2)
    h = case.handle(G, Np, seed=5, burnin=10, n_initial=n0, resample=True, alpha=0.2)
    h.set_history(np.stack([case.theta0(rng, G * Np) for _ in range(n0)]))
    h.set_state(None)
    h.run(n_iter)
    assert h.n_rows == n0 + n_iter
    return h


@pytest.mark.parametrize("centre", [0.0, 1e4])
def test_run_after_prior_rows(backend, centre):
    """resample with n_initial prior rows: a range that straddles the prior rows and the iterations"""
    with _run_after_prior_rows(centre) as h:
        check_diagnostics(h, 25, 50, "prior rows and iterations")
        check_moments(h, 25, 50, "prior rows and iterations")


def test_default_range_is_every_stored_row(backend):
    """moments() and diagnostics() without a range cover every stored row, the n_initial prior rows included, as
    samples() does"""
    with _run_after_prior_rows(0.0) as h:
        s = h.samples()
        cnt, mean, var = h.moments()
        assert cnt == s.shape[0] * s.shape[2]
        for k in range(h.d):
            r_mean, r_var = ref_moments(s[:, k, :])
            assert abs(mean[k] - r_mean) <= TOL_MEAN * max(abs(r_mean), math.sqrt(r_var)), (k, mean[k], r_mean)
            assert abs(var[k] - r_var) <= TOL_VAR * r_var, (k, var[k], r_var)
        assert np.array_equal(h.diagnostics()[0], h.diagnostics(0, h.n_rows)[0])

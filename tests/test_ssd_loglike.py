"""The log-likelihoods of the three models that stream a sum of squared deviations (mvnormal, hier_normal, mvnormal_full)
against an extended-precision reference of the same model, at large data offsets, extreme data and sigma scales,
heavy-tailed rows, the limits of the fixed-point cross term and ill-conditioned covariances.

Every kernel of these models evaluates  SSD = ssd_xx - 2 B + n sum_k m'_k^2  on data centred on a vector c (x' = x - c,
m' = mean - c; mvnormal_full whitens both): ssd_xx comes from k_pack_rows, the cross term B from the DMMA stream
(k_stage_means + k_xdot, k_propose + k_xdot, or k_chunk_persist) on a per-particle fixed-point grid, m' from centred_mean
(de_particle.h), and finalize_ll combines them.  The reference never expands the square: in np.longdouble it sums
(x_ik - mu_k)^2 directly (mvnormal), (y_sj - mu - b_s)^2 (hier_normal, mu + b_s taken exactly) and |L^-1 (x_i - mu)|^2 with
L the Cholesky factor of the covariance in long double (mvnormal_full).  Above SUFFSTAT_N observations it uses the exact
algebra of long-double sufficient statistics instead; both forms, and the reference itself against exact rational /
50-digit arithmetic, are checked here.

Each value is checked against a bound derived from the case (`loglike_bound`), not a blanket tolerance, and so is the
quantity every accept decision rests on, (ll_p - ll_0) - (ref_p - ref_0).  Every check runs on the host-only test double
and, with -m gpu, on the CUDA backend."""
import math
from fractions import Fraction

import numpy as np
import pytest

import common
from common import D

LD = np.longdouble
U = 2.0 ** -53
SUFFSTAT_N = 100_000           # observations per dimension from which the reference uses sufficient statistics
OFFSETS = [0.0, 1e2, -1e2, 1e4, 1e6, 1e8]      # data offsets, in data sd
CONDS = [1e2, 1e6, 1e10]

# Worst over every case of this file (python -m pytest -s prints them), measured on the test double and on one B200
# (1000 W power limit), the same on both: |error| / bound 0.564 for ll and 0.534 for ll_p - ll_0 (hier_normal: the
# rounding of mu + b_s, which both do alike); relative ll error against the long-double reference 8.9e-9 (mvnormal_full
# at condition 1e10: the double Cholesky factor); |(ll_p - ll_0) - (ref_p - ref_0)| 9.8e-6 where |ref_p - ref_0| < 1e3.
WORST = {"ll_ratio": 0.0, "diff_ratio": 0.0, "ll_rel": 0.0, "diff_abs": 0.0}


@pytest.fixture(params=["emu", pytest.param("cuda", marks=pytest.mark.gpu)])
def backend(request):
    """Binds the test double or the CUDA library for one test (the conftest fixtures set each up once per session)."""
    request.getfixturevalue(request.param)
    if request.param == "cuda":
        common.use_cuda()
    else:
        D._ffi.use_library(common.EMU_LIB)
    return request.param


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    yield
    print("\nworst over test_ssd_loglike.py: " + ", ".join(f"{k} {v:.3e}" for k, v in WORST.items()))


# ---- cases -------------------------------------------------------------------------------------------------------------
def _noise(rng, shape, tails):
    if tails == "t1.5":
        return rng.standard_t(1.5, size=shape)
    z = rng.normal(size=shape)
    if tails == "outlier":                 # one row 1e6 times the typical row norm
        z[0] *= 1e6
    return z


def random_cov(rng, k, cond):
    """Q diag Q' with a random orthogonal Q and eigenvalues log-spaced from 1 down to 1 / cond"""
    q, r = np.linalg.qr(rng.normal(size=(k, k)))
    q = q * np.sign(np.diag(r))
    cov = (q * np.geomspace(1.0, 1.0 / cond, k)) @ q.T
    return (cov + cov.T) / 2.0


def make(kind, n, k, rng, offset=0.0, sd=1.0, tails="normal", cond=1e2):
    """One model: data at `offset` data sd from 0 (a different offset per dimension / subject, of the same size) with
    spread sd.  mvnormal: x[n][k]; hier_normal: k subjects x n observations; mvnormal_full: x[n][k] ~ N(mu, sd^2 cov)."""
    shift = offset * sd * (1.0 + 0.5 * rng.uniform(size=k))
    case = dict(kind=kind, n=n, k=k, sd=sd, cov=None)
    if kind == "mvnormal":
        case["x"] = shift + sd * _noise(rng, (n, k), tails)
        case["d"] = k + 1
    elif kind == "hier_normal":
        case["x"] = shift[:, None] + sd * _noise(rng, (k, n), tails)
        case["d"] = k + 3
    else:
        cov = random_cov(rng, k, cond)
        case["cov"] = cov
        case["x"] = shift + sd * (_noise(rng, (n, k), tails) @ np.linalg.cholesky(cov).T)
        case["d"] = k + 1
    d = case["d"]
    case["prior"] = [("flat",)] * d
    case["lo"] = [-np.inf] * d
    case["hi"] = [np.inf] * d
    scale_at = {"mvnormal": [k], "mvnormal_full": [k], "hier_normal": [1, k + 2]}[kind]
    for j in scale_at:
        case["lo"][j] = 0.0
    case["colmean"] = (case["x"].astype(LD).sum(axis=0 if kind != "hier_normal" else 1) / n).astype(float)
    return case


def particles(case, rng, n_spread=6, n_far=3, at_centre=True, sig=1.0):
    """parameter vectors: at posterior spread around the data mean, far from the data (|m'| >> data spread), and one whose
    means are the column means rounded to double (mvnormal_full: the centre its data are whitened on; msq ~ 0)"""
    kind, k, sd, n = case["kind"], case["k"], case["sd"], case["n"]
    c = case["colmean"]
    dev = np.concatenate([rng.normal(size=(n_spread, k)) * sd / math.sqrt(n), rng.normal(size=(n_far, k)) * 1e3 * sd]
                         + ([np.zeros((1, k))] if at_centre else []))
    if kind == "mvnormal_full":
        dev = dev @ np.linalg.cholesky(case["cov"]).T
    P = dev.shape[0]
    sigma = sig * sd * (1.0 + 0.2 * rng.uniform(size=P))
    if kind == "hier_normal":
        mu = np.full(P, c.mean())
        return np.column_stack([mu, np.full(P, sd), (c - mu[:, None]) + dev, sigma])
    return np.column_stack([c + dev, sigma])


# ---- the reference -------------------------------------------------------------------------------------------------------
def chol_ld(S):
    """Cholesky factor in long double"""
    S = np.asarray(S, dtype=LD)
    k = S.shape[0]
    L = np.zeros((k, k), dtype=LD)
    for i in range(k):
        for j in range(i + 1):
            s = S[i, j] - np.dot(L[i, :j], L[j, :j])
            L[i, j] = np.sqrt(s) if i == j else s / L[j, j]
    return L


def solve_lower(L, R):
    """L Z' = R' row by row of R [n][k] (forward substitution, in the dtype of L)"""
    Z = np.zeros(R.shape, dtype=L.dtype)
    for r in range(L.shape[0]):
        Z[:, r] = (R[:, r] - Z[:, :r] @ L[r, :r]) / L[r, r]
    return Z


def engine_factors(cov):
    """the double Cholesky factor, its explicit inverse and log det(cov) exactly as model setup forms them: long-double
    accumulation, each entry rounded to double"""
    k = cov.shape[0]
    L = np.zeros((k, k))
    Li = np.zeros((k, k))
    logdet = 0.0
    for i in range(k):
        for j in range(i + 1):
            s = LD(cov[i, j])
            for q in range(j):
                s -= LD(L[i, q]) * LD(L[j, q])
            if i == j:
                L[i, i] = math.sqrt(float(s))
                logdet += 2.0 * math.log(L[i, i])
            else:
                L[i, j] = float(s / LD(L[j, j]))
    for c in range(k):
        for r in range(c, k):
            t = LD(1) if r == c else LD(0)
            for q in range(c, r):
                t -= LD(L[r, q]) * LD(Li[q, c])
            Li[r, c] = float(t / LD(L[r, r]))
    return L, Li, logdet


def _means_ld(case, th):
    """[P][k] means of the likelihood dimensions in long double (hier_normal: mu + b_s, exact to long double)"""
    th = np.asarray(th, dtype=LD)
    k = case["k"]
    return th[:, :k] if case["kind"] != "hier_normal" else th[:, :1] + th[:, 2:2 + k]


def _obs_major(case):
    x = np.asarray(case["x"], dtype=LD)
    return x.T if case["kind"] == "hier_normal" else x


def quad_forms(case, th, L=None, suffstat=None):
    """sum_i |L^-1 (x_i - m_p)|^2 per parameter vector (L = None: the identity), in long double.  Direct form, or with
    suffstat (default: above SUFFSTAT_N observations) the exact algebra of the sufficient statistics of w_i = L^-1 (x_i - a)
    about a = the column means rounded to double: sum |w|^2 - 2 v.sum w + n |v|^2, v = L^-1 (m_p - a)."""
    X = _obs_major(case)
    M = _means_ld(case, th)
    n = X.shape[0]
    if suffstat is None:
        suffstat = n > SUFFSTAT_N
    whiten = (lambda R: R) if L is None else (lambda R: solve_lower(L, R))
    if not suffstat:
        out = np.zeros(M.shape[0], dtype=LD)
        for p in range(M.shape[0]):
            W = whiten(X - M[p])
            out[p] = (W * W).sum()
        return out
    a = np.asarray(case["colmean"], dtype=LD)
    W = whiten(X - a)
    s1, s2 = W.sum(axis=0), (W * W).sum()
    V = whiten(M - a)
    return s2 - 2 * (V @ s1) + n * (V * V).sum(axis=1)


def loglike_from_q(case, th, Q, logdet=LD(0)):
    """the model's log-likelihood from its quadratic forms, in long double"""
    th = np.asarray(th, dtype=LD)
    k, n = case["k"], case["n"]
    two_pi = LD(2) * LD(np.pi)
    if case["kind"] == "hier_normal":
        s = th[:, k + 2]
        return -LD(n * k) * (np.log(two_pi) / 2 + np.log(s)) - Q / (s * s) / 2
    s = th[:, k]
    return LD(n) * (-(k * np.log(two_pi) + (k * np.log(s * s) + logdet)) / 2) - Q / (s * s) / 2


def reference(case, th):
    """(ref, chol): the exact log-likelihood, and for mvnormal_full the same with the double Cholesky factor the model
    setup uses (the part of the error that rounding the factor of an ill-conditioned covariance to double commits; 0 else)"""
    if case["kind"] != "mvnormal_full":
        ref = loglike_from_q(case, th, quad_forms(case, th))
        return ref, ref
    L = chol_ld(case["cov"])
    ref = loglike_from_q(case, th, quad_forms(case, th, L), 2 * np.log(np.diag(L)).sum())
    Lt, _, logdet_t = engine_factors(case["cov"])
    return ref, loglike_from_q(case, th, quad_forms(case, th, Lt.astype(LD)), LD(logdet_t))


# ---- the bound ---------------------------------------------------------------------------------------------------------
def _split_geometry(k, n):
    """(terms, ksplit_len, qbits) of the streamed kernels' layout (engine.cpp: model setup)"""
    ld = max(64, -(-n // 64) * 64)
    n_ksplit = -(-k // 52)
    ksplit_len = -(-k // n_ksplit)
    terms = ld * n_ksplit
    return terms, ksplit_len, min(50, 62 - max(0, math.ceil(math.log2(terms))))


def quantum(msq, rowmax, qbits):
    """the particle's fixed-point quantum (de_math.h: xd_scale)"""
    b = math.sqrt(msq) * rowmax * 1.0009765625
    if not b < 1e300:
        return math.nan
    e = max(math.frexp(b)[1], -900)
    return math.ldexp(1.0, e - qbits)


def loglike_bound(case, th, suffstat=False):
    """per parameter vector, a bound on |ll - chol| (see `reference`) from the case's own quantities, with N-term sums rounding as
    (8 + sqrt(N)) u of their absolute sum (the error growth of the sequential and blocked orders the kernels use):
      ssd_xx, sum of n k squares of the centred data, and sum_k m'_k^2       (8 + sqrt(N)) u
      B: 2 (terms / 4) q (two rows per rounded chain, |error| <= q / 2 each) + its own sum  A = sum_i sum_k |x'_ik m'_k|
      m'_k: e_k, the rounding of the centred (whitened) mean: u |m'_k|, plus u |mu + b_s| (hier_normal), plus the
            explicit inverse's departure from the factor the data are whitened with (mvnormal_full: cond-dependent)
      sufficient-statistic mode: B is taken as 0; it is n m'.(xbar - c) with c the column means rounded in a sum
    in ll units (/ 2 sigma^2), plus the rounding of the constant part and of the result."""
    kind, k, n = case["kind"], case["k"], case["n"]
    X = _obs_major(case).astype(float)
    c = case["colmean"]
    xc = X - c
    Mld = _means_ld(case, th)
    th = np.asarray(th, dtype=float)
    if kind == "mvnormal_full":
        Lt, Li, _ = engine_factors(case["cov"])
        exact_inv = solve_lower(Lt.astype(LD), np.eye(k, dtype=LD)).T           # rows: (L~^-1)'s rows
        dm = (Mld - np.asarray(c, dtype=LD)).astype(float)                        # mu - c, [P][k]
        xc = solve_lower(Lt, xc)
        mp = dm @ Li.T
        e = np.abs(dm) @ (np.abs(Li - exact_inv.astype(float)).T + (k + 2) * U * np.abs(Li).T) + 2 * U * np.abs(mp)
        sig = th[:, k]
    else:
        mp = (Mld - np.asarray(c, dtype=LD)).astype(float)
        e = U * np.abs(mp)
        if kind == "hier_normal":
            e = e + U * np.abs(Mld.astype(float))
            sig = th[:, k + 2]
        else:
            sig = th[:, k]
    terms, ksplit_len, qbits = _split_geometry(k, n)
    g = lambda N: (8.0 + math.sqrt(N)) * U                                            # noqa: E731
    ssd_xx = float((xc * xc).sum())
    rowmax = 2.0 * math.sqrt(float((xc * xc).sum(axis=1).max()))
    msq = (mp * mp).sum(axis=1)
    A = np.abs(xc).sum(axis=0) @ np.abs(mp).T
    q = np.array([quantum(v, rowmax, qbits) for v in msq])
    ssd = g(n * k) * ssd_xx + 2 * ((terms / 4) * q + g(n * ksplit_len + 4 * ksplit_len * ksplit_len) * A) \
        + n * (g(k) * msq + 2 * (np.abs(mp) * e).sum(axis=1) + (e * e).sum(axis=1))
    if suffstat:
        dc = g(n) * np.abs(c) + np.abs(X.astype(LD).mean(axis=0) - np.asarray(c, dtype=LD)).astype(float)
        ssd = ssd + 2 * n * (np.abs(mp) @ (dc if kind != "mvnormal_full" else np.abs(Li) @ dc))
    n_obs = n * k if kind == "hier_normal" else n
    logdet = abs(engine_factors(case["cov"])[2]) if kind == "mvnormal_full" else 0.0
    const = n_obs * (2.0 * k + 2.0 * k * np.abs(np.log(sig)) + logdet + 2.0)
    return ssd / (2 * sig * sig) + 16 * U * ((ssd_xx + 2 * A + n * msq) / (2 * sig * sig) + const)


def check(case, th, ll, suffstat=False, what=""):
    """ll (float64 [P]) against the reference.  Each value must lie within its bound of the exact log-likelihood with the
    double Cholesky factor (`chol`; mvnormal / hier_normal: the reference itself), and each difference to particle 0
    within the two particles' bounds: so the difference to the long-double reference is within the bound plus what
    rounding the factor to double changes."""
    ref, chol = reference(case, th)
    bound = loglike_bound(case, th, suffstat)
    ll = np.asarray(ll, dtype=float)
    assert np.all(np.isfinite(ll)), what
    err = np.abs(ll.astype(LD) - chol).astype(float)
    ratio = err / bound
    WORST["ll_ratio"] = max(WORST["ll_ratio"], float(ratio.max()))
    WORST["ll_rel"] = max(WORST["ll_rel"], float((np.abs(ll.astype(LD) - ref) / np.abs(ref)).max()))
    assert ratio.max() <= 1.0, (what, int(ratio.argmax()), float(ratio.max()), float(err.max()))
    dref, dchol = ref - ref[0], chol - chol[0]
    derr = np.abs((ll.astype(LD) - ll[0]) - dchol).astype(float)
    dratio = derr / (bound + bound[0])
    near = np.abs(dref.astype(float)) < 1e3                  # differences an accept decision can turn on
    WORST["diff_ratio"] = max(WORST["diff_ratio"], float(dratio.max()))
    WORST["diff_abs"] = max(WORST["diff_abs"], float(np.abs((ll.astype(LD) - ll[0]) - dref).astype(float)[near].max()))
    assert dratio.max() <= 1.0, (what, int(dratio.argmax()), float(dratio.max()), float(derr.max()))


def handle(case, G, Np, **kw):
    h = D.Handle(G, Np, case["d"], case["lo"], case["hi"], **kw)
    extra = dict(cov=case["cov"]) if case["kind"] == "mvnormal_full" else {}
    h.set_model(case["kind"], case["prior"], x=case["x"], **extra)
    return h


def eval_check(case, th, what="", **kw):
    with handle(case, 1, max(3, th.shape[0]), **kw) as h:
        ll = h.eval(th)[0]
    check(case, th, ll, what=what)
    return ll


KINDS = ["mvnormal", "hier_normal", "mvnormal_full"]
SHAPE = {"mvnormal": (200, 7), "hier_normal": (40, 9), "mvnormal_full": (300, 6)}


def _exact(v):
    return Fraction(*LD(v).as_integer_ratio())


# ---- the reference, checked --------------------------------------------------------------------------------------------
def test_reference_against_exact_arithmetic():
    """the long-double reference against rational arithmetic (mvnormal, hier_normal) and 50-digit arithmetic
    (mvnormal_full, mpmath) at one small size, at an offset of 1e8 sd"""
    import mpmath
    rng = np.random.default_rng(1)
    for kind in ("mvnormal", "hier_normal"):
        case = make(kind, 5, 3, rng, offset=1e8)
        th = particles(case, rng, 2, 1)
        Q = quad_forms(case, th, suffstat=False)
        X = _obs_major(case)
        for p, t in enumerate(th):
            m = [Fraction(t[j]) for j in range(3)] if kind == "mvnormal" else [Fraction(t[0]) + Fraction(t[2 + j]) for j in range(3)]
            exact = sum((Fraction(float(X[i, j])) - m[j]) ** 2 for i in range(5) for j in range(3))
            assert abs(_exact(Q[p]) - exact) <= Fraction(2 ** -60) * exact, (kind, p)
    mpmath.mp.dps = 50
    case = make("mvnormal_full", 5, 4, rng, offset=1e4, cond=1e6)
    th = particles(case, rng, 2, 1)
    Q = quad_forms(case, th, chol_ld(case["cov"]), suffstat=False)
    Lm = mpmath.cholesky(mpmath.matrix(case["cov"].tolist()))
    for p, t in enumerate(th):
        exact = mpmath.mpf(0)
        for i in range(5):
            z = mpmath.lu_solve(Lm, mpmath.matrix([mpmath.mpf(case["x"][i, j]) - mpmath.mpf(t[j]) for j in range(4)]))
            exact += sum(v * v for v in z)
        num, den = LD(Q[p]).as_integer_ratio()
        assert abs(mpmath.mpf(num) / den - exact) <= mpmath.mpf(1e-13) * exact, p    # cond 1e6: 1e-19 * 1e6 of room


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("offset", [0.0, 1e4, 1e8])
def test_sufficient_statistics_equal_the_direct_form(kind, offset):
    rng = np.random.default_rng(2)
    n, k = 3000, 5
    case = make(kind, n, k, rng, offset=offset, cond=1e6)
    th = particles(case, rng)
    L = chol_ld(case["cov"]) if kind == "mvnormal_full" else None
    a, b = quad_forms(case, th, L, suffstat=False), quad_forms(case, th, L, suffstat=True)
    assert np.max(np.abs(a - b) / np.abs(a)) <= 1e-15


# ---- demcmc_eval (k_stage_means + k_xdot + k_eval_finish) ----------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("offset", OFFSETS)
@pytest.mark.parametrize("sd", [1e-6, 1.0, 1e6])
def test_eval_at_offsets_and_scales(backend, kind, offset, sd):
    rng = np.random.default_rng(abs(int(offset)) % 1000 + int(-math.log10(sd)) + 7 + KINDS.index(kind))
    case = make(kind, *SHAPE[kind], rng, offset=offset, sd=sd, cond=1e6)
    eval_check(case, particles(case, rng), what=(kind, offset, sd))


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("sig", [1e-3, 1e3])
@pytest.mark.parametrize("offset", [0.0, 1e6])
def test_eval_with_sigma_far_from_the_data_sd(backend, kind, sig, offset):
    rng = np.random.default_rng(11)
    case = make(kind, *SHAPE[kind], rng, offset=offset)
    eval_check(case, particles(case, rng, sig=sig), what=(kind, sig, offset))


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("tails", ["t1.5", "outlier"])
@pytest.mark.parametrize("offset", [0.0, 1e4])
def test_eval_with_heavy_tails(backend, kind, tails, offset):
    """Student-t rows (nu = 1.5) and one row 1e6 times the typical norm: ssd_rowmax, and with it every particle's
    fixed-point quantum, is set by the largest row"""
    rng = np.random.default_rng(12)
    case = make(kind, *SHAPE[kind], rng, offset=offset, tails=tails)
    eval_check(case, particles(case, rng), what=(kind, tails, offset))


# n = 4096 -> 4097: ssd_ld * n_ksplit crosses 2^12 and qbits drops below 50; n = 1, 63, 64, 65: one ragged tile
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", [1, 63, 64, 65, 4096, 4097])
def test_eval_at_the_qbits_limits(backend, kind, n):
    rng = np.random.default_rng(n)
    case = make(kind, n, 3, rng, offset=1e4)
    assert _split_geometry(3, n)[2] == (50 if n <= 4096 else 49)
    eval_check(case, particles(case, rng), what=(kind, n))


@pytest.mark.parametrize("kind", KINDS)
def test_eval_with_a_million_observations(backend, kind):
    """n = 2^20 + 1: qbits = 41, the coarsest grid a single dimension split gets; the reference from sufficient statistics"""
    n = 2 ** 20 + 1
    assert _split_geometry(3, n)[2] == 41
    rng = np.random.default_rng(20)
    case = make(kind, n, 3, rng, offset=1e6)
    eval_check(case, particles(case, rng, 4, 2), what=kind)


# d = 50: half k-step | 52: 13 full k-steps | 7: short split | 3: one k-step | 100: two splits | 110: three splits of 37 |
# hierarchical 1000 subjects x 50: 20 splits
@pytest.mark.parametrize("kind,n,k", [("mvnormal", 130, 50), ("mvnormal", 63, 52), ("mvnormal", 64, 7), ("mvnormal", 200, 3),
                                      ("mvnormal", 65, 100), ("mvnormal", 300, 110), ("hier_normal", 50, 1000),
                                      ("hier_normal", 65, 102), ("mvnormal_full", 130, 50), ("mvnormal_full", 65, 110)])
def test_eval_across_dimension_shapes(backend, kind, n, k):
    rng = np.random.default_rng(n + k)
    case = make(kind, n, k, rng, offset=1e4, cond=1e4)
    eval_check(case, particles(case, rng, 5, 2), what=(kind, n, k))


@pytest.mark.parametrize("cond", CONDS)
@pytest.mark.parametrize("offset", OFFSETS)
def test_full_covariance_conditioning_and_offsets(backend, cond, offset):
    """mvnormal_full: the means are whitened on the device; centred first, so the offset does not cancel there"""
    rng = np.random.default_rng(int(math.log10(cond)) * 31 + OFFSETS.index(offset))
    case = make("mvnormal_full", 2000, 10, rng, offset=offset, cond=cond)
    eval_check(case, particles(case, rng), what=(cond, offset))


@pytest.mark.parametrize("kind", KINDS)
def test_non_finite_means_are_never_accepted(backend, kind):
    """a NaN or infinite mean gives a non-finite log-likelihood, and a proposal built from it is never accepted"""
    rng = np.random.default_rng(13)
    case = make(kind, *SHAPE[kind], rng, offset=1e4)
    th = particles(case, rng, 4, 0, at_centre=False)
    j = 2 if kind == "hier_normal" else 0
    for bad in (np.nan, np.inf, -np.inf):
        t = th.copy()
        t[1, j] = bad
        with handle(case, 1, 4) as h:
            ll = h.eval(t)[0]
        assert not np.isfinite(ll[1]) and np.all(np.isfinite(ll[[0, 2, 3]])), (bad, ll)
    G, Np = 2, 8
    th0 = particles(case, rng, G * Np, 0, at_centre=False)
    th0[3, j] = np.nan
    th0[9, j] = np.inf
    with handle(case, G, Np, seed=4, burnin=2, trace=True) as h:
        h.set_state(th0)
        h.run(3)
        tr = h.trace()
    prop = tr["prop_theta"]
    nonfinite = ~np.all(np.isfinite(prop), axis=2)
    assert nonfinite.any()
    assert not np.isfinite(tr["prop_weight"][nonfinite]).any()
    assert not tr["accepted"][nonfinite].any()


# ---- every proposal of a native run (k_propose + k_xdot + k_accept, or k_chunk_persist) ---------------------------------
@pytest.mark.parametrize("persist", ["1", "0"])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("offset", [0.0, 1e4, 1e8])
def test_every_proposal_of_a_run(backend, kind, offset, persist, monkeypatch):
    monkeypatch.setenv("DEMCMC_PERSIST", persist)
    rng = np.random.default_rng(14)
    n, k = (130, 50) if kind == "mvnormal" else (40, 60) if kind == "hier_normal" else (300, 8)
    case = make(kind, n, k, rng, offset=offset, cond=1e6)
    G, Np = 4, 24
    th0 = particles(case, rng, G * Np, 0, at_centre=False)
    with handle(case, G, Np, seed=5, burnin=2, trace=True, theta_snooker=0.1, alpha=0.2) as h:
        h.set_state(th0)
        h.run(3)
        tr = h.trace()
        ctr = h.counters()
    if backend == "cuda":
        assert (ctr["persistent_chunks"] > 0) == (persist == "1"), ctr
    th = tr["prop_theta"].reshape(-1, case["d"])
    w = tr["prop_weight"].reshape(-1)
    inb = np.all((th >= case["lo"]) & (th <= case["hi"]), axis=1)
    assert inb.sum() > 0.9 * th.shape[0]
    check(case, th[inb], w[inb], what=(kind, offset, persist))          # flat priors: the weight is the log-likelihood


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("offset", [1e4, 1e8])
def test_sufficient_stat_mode_at_offsets(backend, kind, offset):
    """demcmc_set_sufficient_stat: B taken as 0 on data centred on their column means"""
    rng = np.random.default_rng(15)
    case = make(kind, *SHAPE[kind], rng, offset=offset, cond=1e6)
    th = particles(case, rng)
    with handle(case, 1, th.shape[0]) as h:
        h.set_sufficient_stat(True)
        ll = h.eval(th)[0]
    check(case, th, ll, suffstat=True, what=(kind, offset))


@pytest.mark.parametrize("kind", KINDS)
def test_two_device_handle(backend, kind):
    if backend == "cuda" and D._ffi.lib().demcmc_device_count() < 2:
        pytest.skip("needs two GPUs")
    rng = np.random.default_rng(16)
    case = make(kind, *SHAPE[kind], rng, offset=1e4, cond=1e6)
    th = particles(case, rng)
    G, Np = 4, 8
    with handle(case, G, Np, devices=[0, 1]) as h:
        check(case, th, h.eval(th)[0], what=kind)
    th0 = particles(case, rng, G * Np, 0, at_centre=False)
    with handle(case, G, Np, seed=6, burnin=2, trace=True, devices=[0, 1]) as h:
        h.set_state(th0)
        h.run(2)
        tr = h.trace()
    pt = tr["prop_theta"].reshape(-1, case["d"])
    w = tr["prop_weight"].reshape(-1)
    inb = np.all((pt >= case["lo"]) & (pt <= case["hi"]), axis=1)
    check(case, pt[inb], w[inb], what=kind)

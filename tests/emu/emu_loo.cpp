// emu_loo.cpp -- host versions of the model-comparison launchers of csrc/backend.h (launch_pointwise, launch_psis),
// for the host-only test double.
//
// Test infrastructure, not a product path: tests/test_loo.py compiles this file together with tests/emu/emu_backend.cpp,
// csrc/engine.cpp and csrc/planner.cpp into a test double of its own.  The two launchers are declared weak in backend.h,
// so the plain test double (tests/emu/Makefile), which does not define them, still loads and refuses demcmc_loo /
// demcmc_eval_pointwise with DEMCMC_EUNSUPPORTED.  Each function honours the contract of the CUDA kernel it stands for
// (k_ll_obs, k_psis) and is built on the same de_math.h / de_particle.h functions; the sums run serially.
#include <math.h>
#include <algorithm>
#include <utility>
#include <vector>

#include "backend.h"
#include "de_particle.h"

namespace de {
namespace be {

// contract of k_ll_obs: out[i][n], observation-major
int launch_pointwise(const ModelDev &m, const double *theta, int64_t n, int64_t obs0, int64_t n_obs, double *out)
{
    const double *sg = m.has_sigma ? m.sigma_acc : nullptr;
    for (int64_t s = 0; s < n; ++s) {
        const double *th = theta + (size_t)s * m.d;
        double par[MAX_ACC + 5], c0 = 0.0, s2 = 0.0;
        if (m.kind == M_GAUSSIAN) { par[0] = th[0]; par[1] = th[1]; par[2] = log(th[1]); }
        else if (m.kind == M_LNR) { for (int r = 0; r <= m.n_dim; ++r) par[r] = th[r]; }
        else if (m.kind == M_LBA) {
            double pneg = 1.0;
            for (int r = 0; r < m.n_dim; ++r) { par[r] = th[r]; pneg *= norm_cdf(-th[r]); }
            par[m.n_dim] = th[m.n_dim]; par[m.n_dim + 1] = th[m.n_dim + 1]; par[m.n_dim + 2] = th[m.n_dim + 2];
            par[m.n_dim + 3] = 1.0 / (1.0 - pneg);
        } else if (is_ssd(m.kind)) ssd_obs_const(m, th, c0, s2);
        for (int64_t o = 0; o < n_obs; ++o) {
            const int64_t i = obs0 + o;
            double v;
            switch (m.kind) {
            case M_GAUSSIAN: v = gaussian_obs(par, m.x[i]); break;
            case M_LNR: v = lnr_obs(par, m.n_dim, sg, m.x[i], m.choice[i] - 1); break;
            case M_LBA: v = lba_obs(par, m.n_dim, par[m.n_dim + 3], m.lba_floor, m.x[i], m.choice[i] - 1); break;
            case M_BINOMIAL: v = binomial_ll(m.binom_N, m.binom_k, th[0]); break;
            case M_HIER: {
                const int subj = (int)(i / m.n_per);
                const double dl = m.xT[(int64_t)subj * m.ssd_ld + (i - (int64_t)subj * m.n_per)] - centred_mean(m, th, subj);
                v = ssd_obs_ll(c0, s2, dl * dl);
                break;
            }
            case M_MVNORMAL: case M_MVN_FULL: {
                double q = 0.0;
                for (int k = 0; k < m.ssd_k; ++k) { const double dl = m.xT[(int64_t)k * m.ssd_ld + i] - centred_mean(m, th, k); q += dl * dl; }
                v = ssd_obs_ll(c0, s2, q);
                break;
            }
            default: return -1;                       // (the engine refuses models without observations first)
            }
            out[(size_t)o * n + s] = v;
        }
    }
    return 0;
}

// contract of k_psis, one observation after the other (the same estimator, serial sums)
static void psis_one(const double *ll, int S, double *elpd, double *khat, double *lppd, double *p_waic)
{
    double mn = inf(), mx = -inf(), sum = 0.0;
    for (int s = 0; s < S; ++s) {
        if (!isfinite(ll[s])) { *elpd = *khat = *lppd = *p_waic = qnan(); return; }
        mn = std::min(mn, ll[s]); mx = std::max(mx, ll[s]); sum += ll[s];
    }
    double e = 0.0;
    for (int s = 0; s < S; ++s) e += exp(ll[s] - mx);
    *lppd = mx + log(e) - log((double)S);
    const double mean = sum / (double)S;
    double q = 0.0;
    for (int s = 0; s < S; ++s) { const double dl = ll[s] - mean; q += dl * dl; }
    *p_waic = q / (double)(S - 1);
    // log ratios -ll shifted by their maximum, the (M+1)-th largest as the cutoff, the tail above it in (value, draw) order
    std::vector<double> x(S);
    for (int s = 0; s < S; ++s) x[s] = mn - ll[s];
    const int M = psis_tail_len(S);
    std::vector<double> srt(x);
    std::sort(srt.begin(), srt.end());
    const double cutoff = std::max(srt[S - 1 - M], DE_LOG_DBL_MIN);
    std::vector<std::pair<double, int>> tail;
    for (int s = 0; s < S; ++s) if (x[s] > cutoff) tail.push_back({ x[s], s });
    std::sort(tail.begin(), tail.end());
    const int nt = (int)tail.size();
    double k = inf();
    if (nt > 4) {
        const double ec = exp(cutoff);
        std::vector<double> y(nt);
        for (int i = 0; i < nt; ++i) y[i] = exp(tail[i].first) - ec;
        const int m = gpd_grid_len(nt);
        std::vector<double> b(m), prof(m), w(m);
        for (int j = 0; j < m; ++j) {
            b[j] = gpd_grid_b(j, m, y[gpd_quartile_index(nt)], y[nt - 1]);
            double kb = 0.0;
            for (int i = 0; i < nt; ++i) kb += log1p(-b[j] * y[i]);
            prof[j] = gpd_profile(b[j], kb / (double)nt, nt);
        }
        double W = 0.0;
        for (int j = 0; j < m; ++j) {
            double a = 0.0;
            for (int l = 0; l < m; ++l) a += exp(prof[l] - prof[j]);
            w[j] = 1.0 / a;
            if (w[j] >= 10.0 * 2.220446049250313e-16) W += w[j];
        }
        double bp = 0.0;
        for (int j = 0; j < m; ++j) if (w[j] >= 10.0 * 2.220446049250313e-16) bp += b[j] * (w[j] / W);
        double kp = 0.0;
        for (int i = 0; i < nt; ++i) kp += log1p(-bp * y[i]);
        kp /= (double)nt;
        const double sigma = -kp / bp;
        k = gpd_k_prior(kp, nt);
        if (isfinite(k))
            for (int i = 0; i < nt; ++i) {
                double t = log(gpd_inv(((double)i + 0.5) / (double)nt, k, sigma) + ec);
                if (t > 0.0) t = 0.0;
                x[tail[i].second] = t;
            }
    }
    *khat = k;
    double xm = -inf();
    for (int s = 0; s < S; ++s) xm = std::max(xm, x[s]);
    double se = 0.0;
    for (int s = 0; s < S; ++s) se += exp(x[s] - xm);
    const double lse = xm + log(se);
    double tm = -inf();
    for (int s = 0; s < S; ++s) tm = std::max(tm, (x[s] - lse) + ll[s]);
    double st = 0.0;
    for (int s = 0; s < S; ++s) st += exp(((x[s] - lse) + ll[s]) - tm);
    *elpd = tm + log(st);
}

int launch_psis(const double *ll, int64_t n_draws, int64_t n_obs, double *elpd, double *khat, double *lppd, double *p_waic)
{
    for (int64_t i = 0; i < n_obs; ++i) psis_one(ll + (size_t)i * n_draws, (int)n_draws, elpd + i, khat + i, lppd + i, p_waic + i);
    return 0;
}

} // namespace be
} // namespace de

// de_particle.h -- the per-particle parts of the population step (proposal, bounds, prior,
// Metropolis accept, state write), written once against a "cooperating lanes" policy C:
//   C::lane(), C::width()      this lane and the number of lanes sharing one particle
//   C::sum(x)                  sum over lanes, same value returned to every lane, fixed order
//   C::all(b)                  logical AND over lanes
//   C::min_int(i)              minimum over lanes
//   C::sync()                  makes the lanes' global-memory writes visible to each other
//   C::dependency_wait()       called once, before the first access to state written by an earlier
//                              kernel (programmatic dependent launch); a no-op on the host
// kernels.cu instantiates it with a 32-lane warp; the host test double with a single lane.
#pragma once
#include "de_types.h"

namespace de {

struct SerialLanes {
    DE_HD int lane() const { return 0; }
    DE_HD int width() const { return 1; }
    DE_HD double sum(double x) const { return x; }
    DE_HD bool all(bool b) const { return b; }
    DE_HD int min_int(int x) const { return x; }
    DE_HD void sync() const {}
    DE_HD void dependency_wait() const {}
};

// What a backend wants to do with every element of a proposal while it is still in a register
// (kernels.cu stages the likelihood kernel's operands there); the host test double does nothing.
struct NullSink {
    DE_HD void prefetch(int, int) {}
    DE_HD void elem(int, int, double) {}
};
constexpr int PROP_PRE = 2;   // elements per lane whose state-independent inputs are fetched before the dependency wait

// M_MVN_FULL: the whitened mean nu_k = sum_{j <= k} Linv[k][j] (mu_j - c_j), subtracted before the product so that the
// offset of the data does not cancel.  Out of line on the device: the kernels that serve the other kinds as well (eval,
// the persistent chunk kernel) keep their registers for those.
#if defined(__CUDACC__)
__host__ __device__ __noinline__
#else
inline
#endif
double whitened_mean(const double *linv, const double *raw_center, int n_dim, const double *theta, int k)
{
    const double *row = linv + (size_t)k * n_dim;
    double nu = 0.0;
    for (int j = 0; j <= k; ++j) nu += row[j] * (theta[j] - raw_center[j]);
    return nu;
}

// mean of dimension k of the MVN / hierarchical likelihood, relative to the data centre
DE_HD double centred_mean(const ModelDev &m, const double *theta, int k)
{
    if (m.kind == M_MVN_FULL) return whitened_mean(m.linv, m.raw_center, m.n_dim, theta, k) - m.center[k];
    return (m.kind == M_HIER ? theta[0] + theta[2 + k] : theta[k]) - m.center[k];
}

// sum_k mean'_k^2 (the particle-only term of the expanded sum of squares)
template <class C>
DE_HD double mean_sq(const C &co, const ModelDev &m, const double *theta)
{
    if (!is_ssd(m.kind)) return 0.0;
    double s = 0.0;
    for (int k = co.lane(); k < m.ssd_k; k += co.width()) { const double v = centred_mean(m, theta, k); s += v * v; }
    return co.sum(s);
}

// log-likelihood from the reduced kernel output `total`: the sum of per-observation log densities
// for the pointwise kernels; for MVN / hierarchical normal the cross term B = sum_i sum_k x'_ik m'_k
// of the expanded sum of squares  SSD = sum x'^2 - 2 B + n sum_k m'_k^2  (x', m' centred)
DE_HD double finalize_ll(const ModelDev &m, const double *theta, double total, double msq)
{
    switch (m.kind) {
    case M_MVNORMAL: {
        // Multivariate_Guassian_Example.jl:31-33: per column -(d*log2pi + d*log(s^2))/2 - sqmahal/2
        const double ssd = (m.ssd_xx - 2.0 * total) + (double)m.ssd_n * msq;
        const double sig = theta[m.n_dim], s2 = sig * sig, dm = (double)m.n_dim;
        const double c0 = -(dm * DE_LOG2PI + dm * log(s2)) / 2.0;
        return (double)m.n_obs * c0 - (ssd / s2) / 2.0;
    }
    case M_MVN_FULL: {
        // sum(logpdf(MvNormal(mu, sigma^2 * Sigma), data)), Sigma known (SURVEY 8f-4): per column
        // -(k log2pi + logdet(sigma^2 Sigma)) / 2 - sqmahal / 2, sqmahal = |Linv (x - mu)|^2 / sigma^2
        const double ssd = (m.ssd_xx - 2.0 * total) + (double)m.ssd_n * msq;
        const double sig = theta[m.n_dim], s2 = sig * sig, dm = (double)m.n_dim;
        const double c0 = -(dm * DE_LOG2PI + (dm * log(s2) + m.logdet)) / 2.0;
        return (double)m.n_obs * c0 - (ssd / s2) / 2.0;
    }
    case M_HIER: {
        // Hierarchical_Example.jl:36-44: sum_s sum_j logpdf(Normal(0,sigma), y_sj - (mu + b_s))
        const double ssd = (m.ssd_xx - 2.0 * total) + (double)m.ssd_n * msq;
        const double sig = theta[m.n_dim + 2];
        return -(double)m.n_obs * (DE_LOG2PI / 2.0 + log(sig)) - (ssd / (sig * sig)) / 2.0;
    }
    case M_BINOMIAL: return binomial_ll(m.binom_N, m.binom_k, theta[0]);
    case M_RASTRIGIN: {     // test/optimization_tests.jl:15-23
        double y = 10.0 * (double)m.d;
        for (int i = 0; i < m.d; ++i) y += +(theta[i] * theta[i]) - 10.0 * cos(2.0 * DE_PI * theta[i]);
        return y;
    }
    default: return total;
    }
}

// one observation of the MVN / hierarchical kinds (demcmc_eval_pointwise): the log density is c0 - (q / s2) / 2, q the
// squared distance of the centred observation from the centred mean -- finalize_ll's terms for a single observation
DE_HD void ssd_obs_const(const ModelDev &m, const double *theta, double &c0, double &s2)
{
    const double dm = (double)m.n_dim;
    if (m.kind == M_HIER) {
        const double sig = theta[m.n_dim + 2];
        s2 = sig * sig;
        c0 = -(DE_LOG2PI / 2.0 + log(sig));
        return;
    }
    const double sig = theta[m.n_dim];
    s2 = sig * sig;
    c0 = m.kind == M_MVN_FULL ? -(dm * DE_LOG2PI + (dm * log(s2) + m.logdet)) / 2.0 : -(dm * DE_LOG2PI + dm * log(s2)) / 2.0;
}
DE_HD double ssd_obs_ll(double c0, double s2, double q) { return c0 - (q / s2) / 2.0; }

// in_bounds (utilities.jl:70-78) + prior_loglike of one parameter vector
template <class C>
DE_HD void bounds_and_prior(const C &co, const ConfigDev &cfg, const ModelDev &m, const double *theta, bool &inb, double &prior)
{
    bool ok = true;
    double ps = 0.0;
    for (int k = co.lane(); k < cfg.d; k += co.width()) {
        const double v = theta[k];
        ok = ok && (v >= cfg.lo[k] && v <= cfg.hi[k]);
        const Prior pr = m.prior[k];
        ps += prior_elem(pr, v, pr.kind == PRIOR_NORMAL_REF ? theta[pr.ref] : 0.0);
    }
    inb = co.all(ok);
    prior = co.sum(ps);
}

// the state-independent draws of the update of local position p in this sweep (native mode)
DE_HD PlanRec make_plan(const ConfigDev &cfg, const SweepCtx &ctx, int p)
{
    const int Np = cfg.Np;
    const int g = p / Np, j = p - g * Np;
    const uint32_t unit = (uint32_t)((cfg.group_begin + g) * Np + j);
    const bool mutate = ctx.mutate[g] != 0;
    PlanRec r;
    r.i0 = r.i1 = r.i2 = r.hr0 = r.hr1 = r.hr2 = -1; r.pad = 0; r.g1 = 0.0; r.g2 = 0.0;
    if (cfg.resample) {
        const PlanHist pl = plan_particle_hist(cfg.seed, ctx.sweep, unit, mutate, cfg.theta_snooker, ctx.donor_rows, (int64_t)cfg.P_hist);
        r.kind = pl.kind; r.i0 = pl.id[0]; r.i1 = pl.id[1]; r.i2 = pl.id[2]; r.hr0 = pl.row[0]; r.hr1 = pl.row[1]; r.hr2 = pl.row[2]; r.u_base = pl.u_base;
    } else {
        const Plan pl = plan_particle(cfg.seed, ctx.sweep, unit, j, Np, mutate, cfg.theta_snooker);
        r.kind = pl.kind; r.i0 = pl.i0; r.i1 = pl.i1; r.i2 = pl.i2; r.u_base = pl.u_base;
    }
    if (r.kind != KIND_MUTATION) { const dbl2 gg = gamma_draw(cfg.seed, ctx.sweep, unit, r.kind, cfg.proposal, ctx.in_burnin != 0, cfg.d); r.g1 = gg.a; r.g2 = gg.b; }
    r.u_acc = uniform2(cfg.seed, ST_ACC, ctx.sweep, unit, 0).a;
    return r;
}

// a record drawn by an earlier launch: read past the (non-coherent) L1, four 16-byte loads
DE_HD PlanRec load_plan(const PlanRec *r)
{
#if defined(__CUDA_ARCH__)
    union { PlanRec rec; int4 q[4]; } u;
    const int4 *src = reinterpret_cast<const int4 *>(r);
    u.q[0] = __ldcg(src); u.q[1] = __ldcg(src + 1); u.q[2] = __ldcg(src + 2); u.q[3] = __ldcg(src + 3);
    return u.rec;
#else
    return *r;
#endif
}

DE_HD double load_plan_uacc(const PlanRec *r)
{
#if defined(__CUDA_ARCH__)
    return __ldcg(&r->u_acc);
#else
    return r->u_acc;
#endif
}

// crossover!(model,de,group,pt[,block]) / mutation! up to evaluate_fitness!: writes the proposal,
// its prior, bounds flag and snooker adjustment (crossover.jl:30-99,154-273,301-352; mutation.jl:13-25)
template <class C, class S>
DE_HD void propose_particle(const C &co, const ConfigDev &cfg, const ModelDev &m, const SweepCtx &ctx, int p, S &sink)
{
    const int Np = cfg.Np, d = cfg.d;
    const int g = p / Np, j = p - g * Np;
    const uint32_t unit = (uint32_t)((cfg.group_begin + g) * Np + j);
    const double *tcur = ctx.cur_theta + (size_t)p * d;
    double *prop = ctx.prop_theta + (size_t)p * d;

    int kind, i0 = -1, i1 = -1, i2 = -1, hr0 = -1, hr1 = -1, hr2 = -1;
    double g1 = 0.0, g2 = 0.0, u_base = 0.0;
    if (ctx.replay) {
        kind = ctx.t_kind[p];
        i0 = ctx.t_idx[p * 3]; i1 = ctx.t_idx[p * 3 + 1]; i2 = ctx.t_idx[p * 3 + 2];
        if (cfg.resample) { hr0 = ctx.t_idx_row[p * 3]; hr1 = ctx.t_idx_row[p * 3 + 1]; hr2 = ctx.t_idx_row[p * 3 + 2]; }
        g1 = ctx.t_g1[p]; g2 = ctx.t_g2[p];
    } else {
        const PlanRec pl = ctx.plan ? load_plan(ctx.plan + p) : make_plan(cfg, ctx, p);
        kind = pl.kind; i0 = pl.i0; i1 = pl.i1; i2 = pl.i2; hr0 = pl.hr0; hr1 = pl.hr1; hr2 = pl.hr2; u_base = pl.u_base; g1 = pl.g1; g2 = pl.g2;
    }
    // everything an element needs that does not depend on the state -- its noise draw, bounds, prior
    // spec -- is fetched for the first PROP_PRE elements of the lane before the dependency wait
    const bool is_mut = kind == KIND_MUTATION;
    auto noise_at = [&](int k) { return ctx.replay ? ctx.t_noise[(size_t)p * d + k] : noise_elem(cfg.seed, ctx.sweep, unit, k, is_mut, cfg.eps, cfg.sigma); };
    double pre_nz[PROP_PRE], pre_lo[PROP_PRE], pre_hi[PROP_PRE];
    Prior pre_pr[PROP_PRE];
DE_PRAGMA_UNROLL
    for (int q = 0; q < PROP_PRE; ++q) {
        const int k = co.lane() + q * co.width();
        pre_nz[q] = 0.0; pre_lo[q] = 0.0; pre_hi[q] = 0.0; pre_pr[q].kind = PRIOR_FLAT;
        if (k < d) { pre_nz[q] = (ctx.block >= 0 && !is_mut && !cfg.blocks[(size_t)ctx.block * d + k]) ? 0.0 : noise_at(k); pre_lo[q] = cfg.lo[k]; pre_hi[q] = cfg.hi[k]; pre_pr[q] = m.prior[k]; sink.prefetch(q, k); }
    }
    co.dependency_wait();
    // a donor that sits before the target in the sweep already holds this sweep's value; with
    const size_t gbase = (size_t)g * Np;
    const size_t P_all = (size_t)cfg.P_hist;
#define DE_SLOT(k) (((k) < j ? ctx.next_theta : ctx.cur_theta) + (gbase + (size_t)(k)) * d)
#define DE_HIST(r, id) (ctx.hist_theta + ((size_t)(r) * P_all + (size_t)ctx.hist_pos[(size_t)(r) * P_all + (size_t)(id)]) * d)
#define DE_DONOR(k, r) (cfg.resample ? DE_HIST(r, k) : DE_SLOT(k))

    double r1 = 0.0, r2 = 0.0;
    const double *pm = nullptr, *pn = nullptr, *pb = nullptr, *pz = nullptr;
    bool has_base = false;
    if (kind == KIND_DE) {
        pm = DE_DONOR(i1, hr1); pn = DE_DONOR(i2, hr2);
        has_base = cfg.proposal == 0 && ctx.in_burnin != 0;
        if (has_base) {
            if (ctx.exact_base) pb = DE_SLOT(i0);                  // select_base always reads the current group
            else {
                // select_base (crossover.jl:282-289) on the sweep-start weights: first slot whose
                // running weight sum is not below u*sum (StatsBase cumulative walk)
                const double *cw = ctx.base_cw + gbase;
                const double t = u_base * ctx.base_tot[g];
                int found = Np - 1;
                for (int q0 = 0; q0 < Np - 1; q0 += co.width()) {
                    const int q = q0 + co.lane();
                    const bool hit = q < Np - 1 && !(cw[q] < t);
                    const int best = co.min_int(hit ? q : 0x7fffffff);
                    if (best != 0x7fffffff) { found = best; break; }
                }
                i0 = found;
                pb = ctx.cur_theta + (gbase + (size_t)i0) * d;
            }
        }
    } else if (kind == KIND_SNOOKER) {
        pz = DE_DONOR(i0, hr0); pm = DE_DONOR(i1, hr1); pn = DE_DONOR(i2, hr2);
        // project (utilities.jl:239-246): v1 = sum(p1.*pd), v2 = sum(pd.^2)
        double v1m = 0.0, v1n = 0.0, v2 = 0.0;
        for (int k = co.lane(); k < d; k += co.width()) {
            const double pd = sub(tcur[k], pz[k]);
            v1m = add(v1m, mul(pm[k], pd));
            v1n = add(v1n, mul(pn[k], pd));
            v2 = add(v2, mul(pd, pd));
        }
        v1m = co.sum(v1m); v1n = co.sum(v1n); v2 = co.sum(v2);
        r1 = v1m / v2; r2 = v1n / v2;
    }
#undef DE_DONOR
#undef DE_HIST
#undef DE_SLOT

    const uint8_t *mask = (ctx.block >= 0 && !is_mut) ? cfg.blocks + (size_t)ctx.block * d : nullptr;
    bool ok = true;
    double sq1 = 0.0, sq2 = 0.0, ps = 0.0;
    const bool one_pass = m.prior_has_ref == 0;                            // no prior reads another parameter
    // An element outside the sweep's block is reset to theta_t,k whatever was proposed for it (reset!,
    // crossover.jl:336-352; a mutation sweep ignores the block, main.jl:205): its noise draw, its donors and the proposal
    // arithmetic are skipped -- the draws are counter-based, so skipping one does not move the others.  With two blocks of
    // 3 and 1000 parameters (Hierarchical_Example.jl:88-92) every other sweep proposes 3 elements instead of 1003.
    auto live = [&](int k) { return !mask || mask[k] != 0; };
    // the lane's first PROP_PRE elements: every operand is requested before any element is computed (a store sits between
    // two elements, so the compiler cannot move the next element's loads above it: the elements' L2 round trips ran one
    // after the other -- with d <= 64 on a warp that is the whole proposal)
    double pre_t[PROP_PRE], pre_m[PROP_PRE], pre_n[PROP_PRE], pre_x[PROP_PRE];
DE_PRAGMA_UNROLL
    for (int q = 0; q < PROP_PRE; ++q) {
        const int k = co.lane() + q * co.width();
        pre_t[q] = 0.0; pre_m[q] = 0.0; pre_n[q] = 0.0; pre_x[q] = 0.0;
        if (k < d) {
            pre_t[q] = tcur[k];
            if (!is_mut && live(k)) {
                if (kind == KIND_DE) { pre_m[q] = pm[k]; pre_n[q] = pn[k]; if (has_base) pre_x[q] = pb[k]; }
            }
            if (kind == KIND_SNOOKER) pre_x[q] = pz[k];
        }
    }
    auto body = [&](int q, int k, double nz, double lo, double hi, const Prior &pr) {
        const bool pre = q < PROP_PRE;
        const double t = pre ? pre_t[q] : tcur[k];
        double v;
        if (!live(k)) v = t;
        else if (is_mut) v = add(t, nz);                                       // utilities.jl:291-298
        else if (kind == KIND_DE) v = de_elem(t, pre ? pre_m[q] : pm[k], pre ? pre_n[q] : pn[k], has_base ? (pre ? pre_x[q] : pb[k]) : t, g1, g2, has_base, nz);
        else v = snooker_elem(t, pre ? pre_x[q] : pz[k], r1, r2, g1, nz);
        if (!is_mut && live(k)) {
            if (cfg.kappa != 1.0) {                                            // recombination! (crossover.jl:301-321)
                const bool keep = ctx.replay ? ctx.t_keep[(size_t)p * d + k] != 0 : keep_elem(cfg.seed, ctx.sweep, unit, k, cfg.kappa);
                if (keep) v = t;
            }
        }
        if (kind == KIND_SNOOKER) {                                            // adjust_loglike (crossover.jl:268-273)
            const double z = pre ? pre_x[q] : pz[k];
            const double a = sub(v, z), b = sub(t, z);
            sq1 = add(sq1, mul(a, a)); sq2 = add(sq2, mul(b, b));
        }
        ok = ok && (v >= lo && v <= hi);
        prop[k] = v;
        if (ctx.tr_theta) ctx.tr_theta[(size_t)p * d + k] = v;
        if (one_pass) ps += prior_elem(pr, v, 0.0);
        sink.elem(q, k, v);
    };
DE_PRAGMA_UNROLL
    for (int q = 0; q < PROP_PRE; ++q) {
        const int k = co.lane() + q * co.width();
        if (k < d) body(q, k, pre_nz[q], pre_lo[q], pre_hi[q], pre_pr[q]);
    }
    // (tried: bounds and prior specs from a table of per-named-parameter segments instead of the per-element arrays, which
    // cost 56 bytes of loads per element; the arrays are L1-resident and the segment lookup cost more than it saved:
    // configs[3] 14.2 vs 14.7 M updates/s)
    for (int k = co.lane() + PROP_PRE * co.width(); k < d; k += co.width()) body(PROP_PRE, k, live(k) ? noise_at(k) : 0.0, cfg.lo[k], cfg.hi[k], m.prior[k]);
    if (!one_pass) {
        co.sync();
        // hierarchical priors: a thousand elements share one sd parameter, so its logarithm is kept
        // (the value normlogpdf would compute, just not a thousand times)
        double ref_sd = qnan(), ref_log = 0.0;
        for (int k = co.lane(); k < d; k += co.width()) {
            const Prior pr = m.prior[k];
            if (pr.kind == PRIOR_NORMAL_REF) {
                const double sd = prop[pr.ref];
                if (!(sd == ref_sd)) { ref_sd = sd; ref_log = log(sd); }
                const double z = (prop[k] - pr.a) / sd;
                ps += -(z * z + DE_LOG2PI) / 2.0 - ref_log;
            } else ps += prior_elem(pr, prop[k], 0.0);
        }
    }
    const bool inb = co.all(ok);
    ps = co.sum(ps);
    double adj = 0.0;
    if (kind == KIND_SNOOKER) { sq1 = co.sum(sq1); sq2 = co.sum(sq2); adj = adjust_loglike(sq1, sq2, d); }
    if (co.lane() == 0) {
        ctx.prop_prior[p] = ps;
        ctx.prop_inb[p] = inb ? 1 : 0;
        ctx.prop_adj[p] = adj;
    }
}

// compute_posterior! tail + mh_update! (utilities.jl:92-99, 201-210) + the row write that replaces
// store_samples! (utilities.jl:161-180).  TEMPER = false compiles the power-posterior terms out (ConfigDev.temp and
// SweepCtx.next_ll must then be NULL): the kernels that are tight on registers take it for untempered handles.
template <class C, bool TEMPER = true>
DE_HD void accept_particle(const C &co, const ConfigDev &cfg, const ModelDev &m, const SweepCtx &ctx, int p)
{
    const int d = cfg.d, Np = cfg.Np;
    const int n_split = m.n_osplit * m.n_ksplit;
    const double *prop = ctx.prop_theta + (size_t)p * d;
    const double *tcur = ctx.cur_theta + (size_t)p * d;
    const int g = p / Np, j = p - g * Np;
    const uint32_t unit = (uint32_t)((cfg.group_begin + g) * Np + j);
    const double u = ctx.replay ? ctx.t_uacc[p] : ctx.plan ? load_plan_uacc(ctx.plan + p) : uniform2(cfg.seed, ST_ACC, ctx.sweep, unit, 0).a;
    co.dependency_wait();
    double total;
    if (is_ssd(m.kind)) total = (double)ctx.ll_acc[p] * ctx.ll_q[p];
    else {
        double part = 0.0;
        if (m.kind != M_BINOMIAL && m.kind != M_RASTRIGIN)
            for (int s = co.lane(); s < n_split; s += co.width()) part += ctx.ll_part[(size_t)p * n_split + s];
        total = co.sum(part);
    }
    const double msq = is_ssd(m.kind) ? ctx.prop_msq[p] : 0.0;
    const double ll = finalize_ll(m, prop, total, msq);
    const bool inb = ctx.prop_inb[p] != 0;
    // compute_posterior! (utilities.jl:92-99), or evaluate_fun! (utilities.jl:113-120): the kernel
    // alone, and out of bounds loses every comparison
    const double wprop = cfg.fitness == FITNESS_FUN ? (inb ? ll : (cfg.update == UPDATE_MAXIMIZE ? -inf() : inf()))
                                                    : (inb ? add(ctx.prop_prior[p], TEMPER ? tempered_ll(cfg, cfg.group_begin + g, ll) : ll) : -inf());
    const double adj = ctx.prop_adj[p];
    const double wcur = ctx.cur_w[p];
    // mh_update! (utilities.jl:201-210), maximize! / minimize! (utilities.jl:212-226)
    const bool acc = cfg.update == UPDATE_MAXIMIZE ? wprop > wcur : cfg.update == UPDATE_MINIMIZE ? wprop < wcur : accept(wprop, wcur, adj, u);
    // (written here, not with the other lane-0 stores below: ll then dies before the row copy, which needs the registers)
    if (TEMPER && ctx.next_ll && co.lane() == 0) ctx.next_ll[p] = acc ? ll : ctx.cur_ll[p];
    double *dst = ctx.next_theta + (size_t)p * d;
    const double *src = acc ? prop : tcur;                     // (uniform over the lanes: only the row that is kept is read)
    {
        double r[PROP_PRE];                                    // (both loads before the first store: one round trip for d <= 2 lanes' widths)
DE_PRAGMA_UNROLL
        for (int q = 0; q < PROP_PRE; ++q) { const int k = co.lane() + q * co.width(); r[q] = k < d ? src[k] : 0.0; }
DE_PRAGMA_UNROLL
        for (int q = 0; q < PROP_PRE; ++q) { const int k = co.lane() + q * co.width(); if (k < d) dst[k] = r[q]; }
    }
    for (int k = co.lane() + PROP_PRE * co.width(); k < d; k += co.width()) dst[k] = src[k];
    if (co.lane() == 0) {
        ctx.next_w[p] = acc ? wprop : wcur;
        ctx.next_id[p] = ctx.cur_id[p];
        if (ctx.next_pos) ctx.next_pos[ctx.cur_id[p] - cfg.group_begin * Np] = p;
        ctx.next_acc[p] = (acc && cfg.update == UPDATE_MH) ? 1 : 0;       // maximize!/minimize! never write Particle.accept
        if (ctx.tr_w) { ctx.tr_w[p] = wprop; ctx.tr_adj[p] = adj; ctx.tr_acc[p] = acc ? 1 : 0; }
        if (ctx.tr_xdot) ctx.tr_xdot[p] = total;
    }
}

} // namespace de

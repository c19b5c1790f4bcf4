// de_math.h -- scalar fp64 building blocks shared by every kernel of libdemcmc_b200 (and by the
// host-side planner, which must draw the same donor indices the kernels draw).
//
// Everything here is __host__ __device__ so the planner and the kernels cannot drift apart.
// Arithmetic that the reference writes as separate Julia operations is kept un-fused
// (de_add/de_mul map to __dadd_rn/__dmul_rn on the device): Julia never contracts a*b+c.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define DE_HD __host__ __device__ __forceinline__
#define DE_PRAGMA_UNROLL _Pragma("unroll")
#else
#define DE_HD inline
#define DE_PRAGMA_UNROLL
#endif

#define DE_LOG2PI 1.8378770664093454835606594728112
#define DE_LOGPI 1.1447298858494001741434273513531
#define DE_PI 3.14159265358979323846264338327950288
#define DE_SQRT1_2 0.70710678118654752440084436210484904
#define DE_INV_SQRT2PI 0.39894228040143267793994605993438187

namespace de {

DE_HD double add(double a, double b)
{
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
DE_HD double sub(double a, double b)
{
#if defined(__CUDA_ARCH__)
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}
DE_HD double mul(double a, double b)
{
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
DE_HD double inf() { return HUGE_VAL; }
DE_HD double qnan() { return HUGE_VAL - HUGE_VAL; }

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon, Moraes, Dror, Shaw 2011) and the draw map
// ---------------------------------------------------------------------------------------------
struct u32x4 { uint32_t x, y, z, w; };

DE_HD uint32_t mulhi32(uint32_t a, uint32_t b)
{
#if defined(__CUDA_ARCH__)
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32);
#endif
}

DE_HD u32x4 philox4x32_10(u32x4 c, uint32_t k0, uint32_t k1)
{
DE_PRAGMA_UNROLL
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = mulhi32(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = mulhi32(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        u32x4 n;
        n.x = hi1 ^ c.y ^ k0; n.y = lo1; n.z = hi0 ^ c.w ^ k1; n.w = lo0;
        c = n;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return c;
}

// streams of the draw map: counter = (k, unit, sweep, stream), key = seed
enum Stream : uint32_t { ST_MIG = 1, ST_MUT = 2, ST_PLAN = 3, ST_GAMMA = 4, ST_NOISE = 5, ST_KAPPA = 6, ST_ACC = 7 };

struct dbl2 { double a, b; };

// two uniforms in [0,1) carrying 53 random bits each (the resolution of Julia's rand())
DE_HD dbl2 uniform2(uint64_t seed, uint32_t stream, uint32_t sweep, uint32_t unit, uint32_t k)
{
    u32x4 c; c.x = k; c.y = unit; c.z = sweep; c.w = stream;
    const u32x4 o = philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    const uint64_t a = ((uint64_t)o.y << 32) | o.x, b = ((uint64_t)o.w << 32) | o.z;
    dbl2 u;
    u.a = (double)(a >> 11) * 0x1.0p-53;
    u.b = (double)(b >> 11) * 0x1.0p-53;
    return u;
}

DE_HD int rand_index(double u, int n) { int i = (int)(u * (double)n); return i >= n ? n - 1 : i; }

// Box-Muller pair scaled to N(0, sigma): elements 2k and 2k+1 of a mutation proposal
DE_HD dbl2 normal2(dbl2 u, double sigma)
{
    const double r = sqrt(-2.0 * log(1.0 - u.a)), ang = 2.0 * DE_PI * u.b;
    double s, c;
#if defined(__CUDA_ARCH__)
    sincos(ang, &s, &c);
#else
    s = sin(ang); c = cos(ang);
#endif
    dbl2 z;
    z.a = 0.0 + sigma * (r * c);
    z.b = 0.0 + sigma * (r * s);
    return z;
}

// noise element k of unit in sweep: b_k ~ Uniform(-eps, eps) (crossover.jl:166-168) or N(0,sigma)
// (mutation.jl:15-18)
DE_HD double noise_elem(uint64_t seed, uint32_t sweep, uint32_t unit, int k, bool mutation, double eps, double sigma)
{
    const dbl2 u = uniform2(seed, ST_NOISE, sweep, unit, (uint32_t)(k >> 1));
    if (mutation) { const dbl2 z = normal2(u, sigma); return (k & 1) ? z.b : z.a; }
    const double uu = (k & 1) ? u.b : u.a;
    return -eps + (eps - (-eps)) * uu;
}

// recombination! (crossover.jl:301-321): rand() <= 1-kappa restores theta_t,k
DE_HD bool keep_elem(uint64_t seed, uint32_t sweep, uint32_t unit, int k, double kappa)
{
    const dbl2 u = uniform2(seed, ST_KAPPA, sweep, unit, (uint32_t)(k >> 1));
    return ((k & 1) ? u.b : u.a) <= (1.0 - kappa);
}

// ---------------------------------------------------------------------------------------------
// the state-independent part of one particle's update: kind and donor slots
// ---------------------------------------------------------------------------------------------
struct Plan { int kind; int i0, i1, i2; double u_base; };
enum { KIND_DE = 0, KIND_SNOOKER = 1, KIND_MUTATION = 2 };

// crossover!(model,de,group,pt) (crossover.jl:30-47): rand() <= theta_snooker picks the branch;
// DE donors = StatsBase.samplepair over group minus Pt (crossover.jl:158-160); snooker donors =
// three distinct slots of the whole group, target included (crossover.jl:241).
DE_HD Plan plan_particle(uint64_t seed, uint32_t sweep, uint32_t unit, int j, int Np, bool mutate, double theta_snooker)
{
    Plan p; p.kind = KIND_MUTATION; p.i0 = p.i1 = p.i2 = -1; p.u_base = 0.0;
    if (mutate) return p;
    const dbl2 u0 = uniform2(seed, ST_PLAN, sweep, unit, 0);
    const dbl2 u1 = uniform2(seed, ST_PLAN, sweep, unit, 1);
    p.u_base = u0.b;
    if (!(u0.a <= theta_snooker)) {
        p.kind = KIND_DE;
        const int n = Np - 1;
        int a = rand_index(u1.a, n), b = rand_index(u1.b, n - 1);
        if (b == a) b = n - 1;
        p.i1 = a >= j ? a + 1 : a;
        p.i2 = b >= j ? b + 1 : b;
    } else {
        p.kind = KIND_SNOOKER;
        const dbl2 u2 = uniform2(seed, ST_PLAN, sweep, unit, 2);
        int a = rand_index(u1.a, Np), b = rand_index(u1.b, Np - 1);
        if (b >= a) ++b;
        int c = rand_index(u2.a, Np - 2);
        const int lo = a < b ? a : b, hi = a < b ? b : a;
        if (c >= lo) ++c;
        if (c >= hi) ++c;
        p.i0 = a; p.i1 = b; p.i2 = c;
    }
    return p;
}

// the same with de.sample = resample (crossover.jl:113-124): the donors are n distinct cells of the
// (rows x ids) view de.samples[1:de.iter-1, 1, :], column-major cell -> (row, id); two by
// StatsBase.samplepair, three distinct for the snooker update.  Cells are 64-bit: rows x ids can
// pass 2^31.
struct PlanHist { int kind; int32_t id[3]; int32_t row[3]; double u_base; };
DE_HD int64_t rand_index64(double u, int64_t n) { int64_t i = (int64_t)(u * (double)n); return i >= n ? n - 1 : i; }
DE_HD PlanHist plan_particle_hist(uint64_t seed, uint32_t sweep, uint32_t unit, bool mutate, double theta_snooker, int64_t ub, int64_t n_ids)
{
    PlanHist p; p.kind = KIND_MUTATION; p.u_base = 0.0;
    for (int q = 0; q < 3; ++q) { p.id[q] = -1; p.row[q] = -1; }
    if (mutate) return p;
    const dbl2 u0 = uniform2(seed, ST_PLAN, sweep, unit, 0);
    const dbl2 u1 = uniform2(seed, ST_PLAN, sweep, unit, 1);
    p.u_base = u0.b;
    const int64_t n = ub * n_ids;
    if (!(u0.a <= theta_snooker)) {
        p.kind = KIND_DE;
        int64_t a = rand_index64(u1.a, n), b = rand_index64(u1.b, n - 1);
        if (b == a) b = n - 1;
        p.row[1] = (int32_t)(a % ub); p.id[1] = (int32_t)(a / ub);
        p.row[2] = (int32_t)(b % ub); p.id[2] = (int32_t)(b / ub);
    } else {
        p.kind = KIND_SNOOKER;
        const dbl2 u2 = uniform2(seed, ST_PLAN, sweep, unit, 2);
        int64_t a = rand_index64(u1.a, n), b = rand_index64(u1.b, n - 1);
        if (b >= a) ++b;
        int64_t c = rand_index64(u2.a, n - 2);
        const int64_t lo = a < b ? a : b, hi = a < b ? b : a;
        if (c >= lo) ++c;
        if (c >= hi) ++c;
        p.row[0] = (int32_t)(a % ub); p.id[0] = (int32_t)(a / ub);
        p.row[1] = (int32_t)(b % ub); p.id[1] = (int32_t)(b / ub);
        p.row[2] = (int32_t)(c % ub); p.id[2] = (int32_t)(c / ub);
    }
    return p;
}

// gamma draws: random_gamma g1 = Uniform(0.5,1), g2 = Uniform(0.5,1) while iter <= burnin else 0
// (crossover.jl:162-164); snooker g = Uniform(1.2,2.2) (crossover.jl:249)
DE_HD dbl2 gamma_draw(uint64_t seed, uint32_t sweep, uint32_t unit, int kind, int proposal, bool in_burnin, int d)
{
    const dbl2 u = uniform2(seed, ST_GAMMA, sweep, unit, 0);
    dbl2 g; g.a = 0.0; g.b = 0.0;
    if (kind == KIND_SNOOKER) { g.a = 1.2 + (2.2 - 1.2) * u.a; return g; }
    if (proposal == 0) { g.a = 0.5 + (1.0 - 0.5) * u.a; g.b = in_burnin ? 0.5 + (1.0 - 0.5) * u.b : 0.0; }
    else if (proposal == 1) g.a = 2.38;
    else g.a = 2.38 / sqrt(2.0 * (double)d);
    return g;
}

// ---------------------------------------------------------------------------------------------
// proposals, element by element
// ---------------------------------------------------------------------------------------------
// random_gamma body (crossover.jl:168): ((t + g1*(m-n)) + g2*(b-t)) + noise, n-ary + folds left;
// fixed/variable gamma (crossover.jl:195,222) drop the base term.
DE_HD double de_elem(double t, double m, double n, double b, double g1, double g2, bool has_base, double noise)
{
    double r = add(t, mul(sub(m, n), g1));
    if (has_base) r = add(r, mul(sub(b, t), g2));
    return add(r, noise);
}

// snooker_update! (crossover.jl:239-257) given r1 = (m.pd)/(pd.pd), r2 = (n.pd)/(pd.pd):
// theta* = (t + g*(pd*r1 - pd*r2)) + noise
DE_HD double snooker_elem(double t, double z, double r1, double r2, double g, double noise)
{
    const double pd = sub(t, z);
    return add(add(t, mul(sub(mul(pd, r1), mul(pd, r2)), g)), noise);
}

// accept (utilities.jl:55-58): p = min(1, exp(w' - w + adj)); rand() <= p; NaN rejects
DE_HD bool accept(double w_prop, double w_cur, double log_adj, double u)
{
    double p = exp(add(sub(w_prop, w_cur), log_adj));
    if (p > 1.0) p = 1.0;
    return u <= p;
}

// adjust_loglike (crossover.jl:268-273) from the two squared norms
// x^n for an integer n >= 0 by squaring: the integer power the reference writes (`norm(...)^(Np - 1)`),
// a dozen multiplications instead of two calls of the general pow() on the slowest proposal of a level
DE_HD double ipow(double x, int n)
{
    double r = 1.0;
    while (n > 0) {
        if (n & 1) r *= x;
        n >>= 1;
        if (n) x *= x;
    }
    return r;
}
DE_HD double adjust_loglike(double sq_prop_z, double sq_t_z, int d)
{
#if defined(__CUDA_ARCH__)
    const double adj1 = ipow(sqrt(sq_prop_z), d - 1);
    const double adj2 = ipow(sqrt(sq_t_z), d - 1);
#else
    const double adj1 = pow(sqrt(sq_prop_z), (double)(d - 1));
    const double adj2 = pow(sqrt(sq_t_z), (double)(d - 1));
#endif
    return log(adj1 / adj2);
}

// ---------------------------------------------------------------------------------------------
// order-independent accumulation of the MVN / hierarchical cross term
// ---------------------------------------------------------------------------------------------
// Every per-row term v = sum_k x'_ik m'_k obeys |v| <= |x'_i| |m'| (Cauchy-Schwarz); a chain of the
// kernel sums two rows, hence rowmax = 2 max_i |x'_i|.  With a per-particle power-of-two quantum
// q = 2^(e - qbits), 2^e > rowmax*|m'|, the value v rounded to a
// multiple of q is an integer below 2^qbits and integer addition is associative: the total does
// not depend on how observations were split over CTAs (level size, GPU count).  The rounding uses
// the classic magic-number add: bits(v + 1.5*2^52*q) - bits(1.5*2^52*q) = round(v/q).
struct XdScale { double magic, q; };
DE_HD XdScale xd_scale(double msq, double rowmax, int qbits)
{
    XdScale s;
    const double bound = sqrt(msq) * rowmax * 1.0009765625;
    if (!(bound < 1e300)) { s.magic = qnan(); s.q = qnan(); return s; }       // means not finite
    int e = 0;
    frexp(bound, &e);                                                          // bound = f * 2^e, f in [0.5, 1)
    if (e < -900) e = -900;
    s.q = ldexp(1.0, e - qbits);
    s.magic = ldexp(1.5, e - qbits + 52);
    return s;
}
DE_HD long long xd_bits(double t)
{
#if defined(__CUDA_ARCH__)
    return __double_as_longlong(t);
#else
    long long b; memcpy(&b, &t, sizeof b); return b;
#endif
}

// ---------------------------------------------------------------------------------------------
// densities
// ---------------------------------------------------------------------------------------------
DE_HD double normlogpdf(double mu, double sigma, double x)
{
    const double z = (x - mu) / sigma;
    return -(z * z + DE_LOG2PI) / 2.0 - log(sigma);
}
DE_HD double norm_cdf(double z) { return 0.5 * erfc(-z * DE_SQRT1_2); }
DE_HD double norm_pdf(double z) { return exp(-0.5 * z * z) * DE_INV_SQRT2PI; }
// log(1 - Phi(z)): direct while erfc is comfortably normal, scaled complement beyond
DE_HD double normlogccdf(double z)
{
    const double x = z * DE_SQRT1_2;
#if defined(__CUDA_ARCH__)
    if (x < 5.0) return log(0.5 * erfc(x));
    return log(0.5 * erfcx(x)) - x * x;
#else
    if (x < 25.0) return log(0.5 * erfc(x));
    const double x2 = x * x;
    double s = 1.0, term = 1.0;
    for (int k = 1; k < 12; ++k) { term *= -(2.0 * k - 1.0) / (2.0 * x2); s += term; }
    return -x2 - log(x) - 0.5 * DE_LOGPI + log(s) - 0.69314718055994530942;
#endif
}

// c0, c1: the parameter-only terms of the log density, computed once on the host (prior_constants)
// so the per-proposal evaluation carries at most one transcendental per element
struct Prior { int32_t kind; int32_t ref; double a, b, c0, c1; };
enum { PRIOR_FLAT = 0, PRIOR_NORMAL = 1, PRIOR_HALFCAUCHY = 2, PRIOR_UNIFORM = 3, PRIOR_BETA = 4, PRIOR_NORMAL_REF = 5 };

inline void prior_constants(Prior &p)
{
    p.c0 = 0.0; p.c1 = 0.0;
    switch (p.kind) {
    case PRIOR_NORMAL: p.c0 = log(p.b); break;
    case PRIOR_HALFCAUCHY: p.c0 = log(p.b); p.c1 = log(1.0 - (atan((0.0 - p.a) / p.b) / DE_PI + 0.5)); break;
    case PRIOR_UNIFORM: p.c0 = log(p.b - p.a); break;
    case PRIOR_BETA: p.c0 = lgamma(p.a) + lgamma(p.b) - lgamma(p.a + p.b); break;
    default: break;
    }
}

// one term of prior_loglike; sd_ref = theta[p.ref] for NORMAL_REF
DE_HD double prior_elem(const Prior &p, double x, double sd_ref)
{
    switch (p.kind) {
    case PRIOR_FLAT: return 0.0;
    case PRIOR_NORMAL: { const double z = (x - p.a) / p.b; return -(z * z + DE_LOG2PI) / 2.0 - p.c0; }
    case PRIOR_NORMAL_REF: return normlogpdf(p.a, sd_ref, x);
    case PRIOR_HALFCAUCHY: {
        if (!(x >= 0.0)) return x != x ? qnan() : -inf();
        const double z = (x - p.a) / p.b;
        return -(log1p(z * z) + DE_LOGPI + p.c0) - p.c1;
    }
    case PRIOR_UNIFORM:
        if (x != x) return qnan();
        return (x >= p.a && x <= p.b) ? -p.c0 : -inf();
    case PRIOR_BETA: {
        if (x != x) return qnan();
        if (!(x >= 0.0 && x <= 1.0)) return -inf();
        const double t1 = (p.a == 1.0) ? 0.0 : (p.a - 1.0) * log(x);
        const double t2 = (p.b == 1.0) ? 0.0 : (p.b - 1.0) * log1p(-x);
        return t1 + t2 - p.c0;
    }
    }
    return qnan();
}

#if defined(__CUDACC__)
// ---- device exp / erfcx for the LBA kernel --------------------------------------------------------------------------
// CUDA's exp() and erfcx() materialise every polynomial coefficient with two UMOVs: in the LBA trial loop a quarter of the
// executed instructions were constant moves and the kernel was ISSUE-bound with the fp64 pipe 65 % busy
// (profiles/r01_v20_k_ll_pointwise_lba_ncu_full_summary.csv).  These two take their coefficients from constant memory as
// operands of the DFMAs.  de_exp_nonpos: exp(x) for x <= 0 (the kernel's arguments are -n^2/2): 2^k * Taylor_13(r),
// |r| <= ln2/2, remainder < 4e-18; below -708 it returns 0 (CUDA returns denormals there: < 1e-307 absolute, far under
// the density floor).  de_erfcx_nonneg: (1 + 2x) erfcx(x) = sum_j c_j t^j, t = (x - 3.75)/(x + 3.75) in [-1, 1)
// (Shepherd & Laframboise 1981; the Chebyshev series of degree 26 fitted with mpmath at 60 digits and converted to the
// monomial basis: max coefficient 1.24, so Horner is well conditioned), one reciprocal for both divisions.  Measured
// against mpmath on [0, 1e8]: <= 2.4 ulp (scipy.special.erfcx: 3.4 ulp); tests/test_device_math.py parses the two tables
// below and repeats that check with the same arithmetic in numpy.
__constant__ double DE_ERFCX_C[27] = {
    1.23751263083782748e+00, -1.40240598585547022e-01, 3.58541548546368986e-03,
    8.22767384901510190e-02, -1.08803930141707458e-01, 9.23043211601983354e-02,
    -5.86933985905476185e-02, 2.83622774215155984e-02, -9.74657954761962327e-03,
    1.75562583242175286e-03, 2.93713594805707372e-04, -2.90153979289867647e-04,
    5.16494077754639890e-05, 2.23839120365506783e-05, -1.14450491258313085e-05,
    -9.72849582211122008e-07, 1.75344342511063340e-06, -5.82628107880077700e-08,
    -2.61147023599009557e-07, 2.42897629254887070e-08, 4.09712231527030054e-08,
    -4.38928415998632824e-09, -6.54556021248026694e-09, 5.45715730470468752e-10,
    9.02214970034058998e-10, -3.75315827795962019e-11, -7.33950500852953997e-11
};
__constant__ double DE_EXP_C[14] = {
    1.0, 1.0, 0.5, 1.0 / 6.0, 1.0 / 24.0, 1.0 / 120.0, 1.0 / 720.0, 1.0 / 5040.0, 1.0 / 40320.0, 1.0 / 362880.0, 1.0 / 3628800.0,
    1.0 / 39916800.0, 1.0 / 479001600.0, 1.0 / 6227020800.0
};
__device__ __forceinline__ double de_exp_nonpos(double x)
{
    const double kd = __dadd_rn(__fma_rn(x, 1.4426950408889634074, 6755399441055744.0), -6755399441055744.0);   // rint(x log2 e)
    double r = __fma_rn(kd, -6.93147180369123816490e-01, x);
    r = __fma_rn(kd, -1.90821492927058770002e-10, r);
    double p = DE_EXP_C[13];
#pragma unroll
    for (int j = 12; j >= 0; --j) p = __fma_rn(p, r, DE_EXP_C[j]);
    const int k = (int)kd;
    const double scale = __hiloint2double((k + 1023) << 20, 0);                      // 2^k, k >= -1022
    return x < -708.0 ? 0.0 : p * scale;                                             // NaN compares false: propagates through p
}
__device__ __forceinline__ double de_erfcx_nonneg(double x)
{
    const double a = x + 3.75, b = __fma_rn(2.0, x, 1.0);
    const double r = 1.0 / (a * b);
    const double t = (x - 3.75) * b * r;
    double p = DE_ERFCX_C[26];
#pragma unroll
    for (int j = 25; j >= 0; --j) p = __fma_rn(p, t, DE_ERFCX_C[j]);
    return x < 4.0e15 ? p * (a * r) : 0.56418958354775628695 / x;                    // beyond: 1 / (x sqrt(pi)); inf -> 0
}
#endif

// ---- per-observation log densities of the "pointwise" kernels ---------------------------------
// Gaussian (Examples/Gaussian_Example.jl:26-28): logpdf(Normal(mu,sigma), x); par = {mu, sigma, log(sigma)}
DE_HD double gaussian_obs(const double *par, double x)
{
    const double z = (x - par[0]) / par[1];
    return -(z * z + DE_LOG2PI) / 2.0 - par[2];
}

// LNR (test/lognormal_race_tests.jl:9-12): winner LogNormal logpdf + losers LogNormal logccdf on
// t - tau; par = {nu[0..nr), tau}; sg = sd per accumulator (NULL => 1)
DE_HD double lnr_obs(const double *par, int nr, const double *sg, double rt, int choice)
{
    const double x = rt - par[nr];
    if (!(x > 0.0)) return x != x ? qnan() : -inf();
    const double lx = log(x);
    double LL = 0.0;
    for (int r = 0; r < nr; ++r) {
        const double s = sg ? sg[r] : 1.0;
        const double z = (lx - par[r]) / s;
        if (r == choice) LL += -(z * z + DE_LOG2PI) / 2.0 - log(s) - lx;
        else LL += normlogccdf(z);
    }
    return LL;
}

// LBA (Examples/Run_LBA.jl:34-37; Brown & Heathcote 2008, sigma = 1): par = {nu[0..na), A, k, tau},
// inv_1mpneg = 1/(1 - prod Phi(-nu_i))
DE_HD double lba_obs(const double *par, int na, double inv_1mpneg, double floor_, double rt, int choice)
{
    const double A = par[na], b = A + par[na + 1], tau = par[na + 2];
    if (rt < tau) return floor_ > 0.0 ? log(floor_) : -inf();
    const double dt = rt - tau;
    double den = 1.0;
#if defined(__CUDA_ARCH__)
    // Device form of the same density, arranged for the fp64 pipe: one division per trial (1/dt; 1/A
    // comes with the particle, par[na+4]) instead of nine, and Phi and phi of each argument share one
    // exponential: phi(n) = e/sqrt(2 pi), Phi(-|n|) = erfcx(|n|/sqrt 2) e / 2 with e = exp(-n^2/2).
    // Differences from the host form are a few ulp (the LBA tolerance of the parity tests is 1e-10).
    const double inv_dt = 1.0 / dt, inv_A = par[na + 4];
    const double q1 = (b - A) * inv_dt, q2 = b * inv_dt;
    for (int r = 0; r < na; ++r) {
        const double v = par[r];
        const double n1 = q1 - v, n2 = q2 - v;
        const double e1 = de_exp_nonpos(-0.5 * n1 * n1), e2 = de_exp_nonpos(-0.5 * n2 * n2);
        const double t1 = 0.5 * de_erfcx_nonneg(fabs(n1) * DE_SQRT1_2) * e1, t2 = 0.5 * de_erfcx_nonneg(fabs(n2) * DE_SQRT1_2) * e2;
        const double c1 = n1 < 0.0 ? t1 : 1.0 - t1, c2 = n2 < 0.0 ? t2 : 1.0 - t2;
        const double p1 = e1 * DE_INV_SQRT2PI, p2 = e2 * DE_INV_SQRT2PI;
        // both forms, then a select: the winner differs from trial to trial, so a warp took both branches anyway (with the
        // divergence bookkeeping on top); the selected value is the one the branch computed
        const double f = (-v * c1 + p1 + v * c2 - p2) * inv_A;
        const double dA = dt * inv_A;
        double F = 1.0 + (n1 * dA) * c1 - (n2 * dA) * c2 + dA * p1 - dA * p2;
        F = F > 0.0 ? F : (F != F ? F : 0.0);
        den *= (r == choice) ? (f > 0.0 ? f : (f != f ? f : 0.0)) : (1.0 - F);
    }
#else
    for (int r = 0; r < na; ++r) {
        const double v = par[r];
        const double n1 = (b - A - dt * v) / dt, n2 = (b - dt * v) / dt;
        const double c1 = norm_cdf(n1), c2 = norm_cdf(n2), p1 = norm_pdf(n1), p2 = norm_pdf(n2);
        if (r == choice) {
            const double f = (-v * c1 + p1 + v * c2 - p2) / A;
            den *= (f > 0.0 ? f : (f != f ? f : 0.0));
        } else {
            double F = 1.0 + ((b - A - dt * v) / A) * c1 - ((b - dt * v) / A) * c2 + (dt / A) * p1 - (dt / A) * p2;
            F = F > 0.0 ? F : (F != F ? F : 0.0);
            den *= (1.0 - F);
        }
    }
#endif
    den = den * inv_1mpneg;
    if (den != den) return -inf();
    if (den < floor_) den = floor_;
    return log(den);
}

// Binomial (test/binomial_tests.jl:15-17): logpdf(Binomial(N,p),k)
DE_HD double binomial_ll(double N, double k, double p)
{
    const double lc = lgamma(N + 1.0) - lgamma(k + 1.0) - lgamma(N - k + 1.0);
    const double a = (k == 0.0) ? 0.0 : k * log(p);
    const double b = (N - k == 0.0) ? 0.0 : (N - k) * log1p(-p);
    return lc + a + b;
}

// ---- Pareto-smoothed importance sampling (include/demcmc_b200.h: demcmc_loo) ----------------------------------------
// The scalar algebra of the generalized-Pareto fit of Zhang & Stephens (2009) as ArviZ's _gpdfit / _gpinv write it, shared
// by k_psis and the host test double.  y[0..n) is the sorted tail, m = 30 + floor(sqrt(n)) grid points.
// grid point j of the fit: b_j = (1 - sqrt(m / (j + 1/2))) / (3 y[q]) + 1 / y[n - 1],  q = floor(n / 4 + 1/2) - 1
DE_HD int gpd_grid_len(int n) { return 30 + (int)sqrt((double)n); }
DE_HD int gpd_quartile_index(int n) { return (int)((double)n / 4.0 + 0.5) - 1; }
DE_HD double gpd_grid_b(int j, int m, double y_q, double y_max)
{
    return (1.0 - sqrt((double)m / ((double)(j + 1) - 0.5))) / (3.0 * y_q) + 1.0 / y_max;
}
// profile log-likelihood of grid point b given kbar = mean_i log1p(-b y_i): n (log(-b / kbar) - kbar - 1)
DE_HD double gpd_profile(double b, double kbar, int n) { return (double)n * (log(-(b / kbar)) - kbar - 1.0); }
// the weakly informative prior on k (ArviZ: prior_k = 10 pseudo-observations at k = 1/2)
DE_HD double gpd_k_prior(double k, int n) { return ((double)n * k + 10.0 * 0.5) / ((double)n + 10.0); }
// GPD quantile at probability p in (0, 1) with shape k and scale sigma
DE_HD double gpd_inv(double p, double k, double sigma)
{
    if (!(sigma > 0.0)) return qnan();
    const double x = fabs(k) < 2.220446049250313e-16 ? -log1p(-p) : expm1(-k * log1p(-p)) / k;
    return x * sigma;
}
// tail length M = ceil(min(S / 5, 3 sqrt(S))) of S draws (r_eff = 1)
DE_HD int psis_tail_len(int S)
{
    const double a = 0.2 * (double)S, b = 3.0 * sqrt((double)S);
    return (int)ceil(a < b ? a : b);
}
#define DE_LOG_DBL_MIN (-708.39641853226410622)   // log(DBL_MIN): the floor of the tail cutoff

} // namespace de

// emu_backend.cpp -- HOST-ONLY TEST DOUBLE of csrc/backend.h.
//
// This is test infrastructure, not a product path: it is compiled only by tests/emu/Makefile into
// tests/emu/libdemcmc_emu.so, and nothing in the package ever loads it (the product library
// fails with DEMCMC_ENODEVICE when there is no CUDA device).  It lets the CPU test-suite exercise
// the engine's host logic (planner levels, row bookkeeping, tape sharding, migration cycle, ABI
// error paths) and the shared __host__ __device__ math in de_math.h / de_particle.h against the
// oracle on a machine without a GPU.  "Device" memory is plain malloc; each "kernel" is a loop
// that honours the same contract as the CUDA kernel of the same name.
#include <math.h>
#include <sched.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>

#include "backend.h"
#include "de_particle.h"

namespace de {
namespace be {

static thread_local std::string g_err;
static thread_local int64_t g_launches = 0;
// exchange hook so a CPU test can stand in for NCCL (tests/test_multirank_gloo.py)
typedef int (*exchange_fn)(int rank, int n, const int *src_rank, const int *dst_rank, double *send, double *recv, int row_len, void *user);
static exchange_fn g_exchange = nullptr;
static void *g_exchange_user = nullptr;

const char *name() { return "emu"; }
const char *last_error() { return g_err.c_str(); }
int device_count() { return 1; }
int set_device(int) { return 0; }
void *dmalloc(size_t b) { return calloc(1, b ? b : 8); }
void dfree(void *p) { free(p); }
void *dmalloc_shared(size_t b) { return calloc(1, b ? b : 8); }
void dfree_shared(void *p) { free(p); }
void *hmalloc_pinned(size_t b) { return calloc(1, b ? b : 8); }
void hfree_pinned(void *p) { free(p); }
int h2d(void *d, const void *s, size_t b) { if (b) memcpy(d, s, b); return 0; }
int d2h(void *d, const void *s, size_t b) { if (b) memcpy(d, s, b); return 0; }
int d2d(void *d, const void *s, size_t b) { if (b) memmove(d, s, b); return 0; }
int dzero(void *d, size_t b) { if (b) memset(d, 0, b); return 0; }
int sync() { return 0; }
void set_lane(int) {}
int lane_fork(int) { return 0; }
int lane_join(int) { return 0; }
void *event_create() { return malloc(8); }
void event_destroy(void *e) { free(e); }
int event_record(void *) { return 0; }
int event_wait(void *) { return 0; }
void *tevent_create() { return malloc(8); }
void tevent_destroy(void *e) { free(e); }
int tevent_elapsed(void *, void *, double *ms) { *ms = 0.0; return 0; }
int dfill(void *d, int v, size_t b) { if (b) memset(d, v, b); return 0; }
int timer_start() { return 0; }
int timer_stop(double *ms) { *ms = 0.0; return 0; }
int64_t launch_count() { return g_launches; }
void timeline_dump() {}

struct ksum_t { double s, c; };
static void kadd(ksum_t &k, double x)
{
    const double t = k.s + x;
    if (isfinite(t)) { if (fabs(k.s) >= fabs(x)) k.c += (k.s - t) + x; else k.c += (x - t) + k.s; }
    k.s = t;
}
static double kval(const ksum_t &k) { return isfinite(k.s) ? k.s + k.c : k.s; }

size_t pack_ssd_doubles(const ModelDev &m) { return (size_t)m.ssd_k * (size_t)m.ssd_ld; }

int launch_pack_ssd(const double *x, int, const double *center_host, ModelDev *m)
{
    ++g_launches;
    double *xT = const_cast<double *>(m->xT), *center = const_cast<double *>(m->center);
    double xx = 0.0;
    for (int k = 0; k < m->ssd_k; ++k) {
        auto at = [&](int64_t i) { return m->kind != M_HIER ? x[i * m->ssd_k + k] : x[(int64_t)k * m->ssd_n + i]; };
        double s = 0.0;
        for (int64_t i = 0; i < m->ssd_n; ++i) s += at(i);
        const double c = center_host ? center_host[k] : (m->ssd_n > 0 ? s / (double)m->ssd_n : 0.0);
        center[k] = c;
        double q = 0.0;
        for (int64_t i = 0; i < m->ssd_ld; ++i) {
            double v = 0.0;
            if (i < m->ssd_n) { v = at(i) - c; q += v * v; }
            xT[(int64_t)k * m->ssd_ld + i] = v;
        }
        xx += q;
    }
    m->ssd_xx = xx;
    m->ssd_rowmax = 0.0;                      // the fixed-point scale is a CUDA-kernel detail
    return 0;
}

// contract of k_xdot / k_ll_pointwise: part[p][split] for every particle of the level
// (MVN / hierarchical: the cross term is handed over as ll_acc = 1, ll_q = the sum)
static int loglik_impl(const ModelDev &m, const double *theta, const Level &lv, double *part)
{
    ++g_launches;
    if (m.kind == M_BINOMIAL || m.kind == M_RASTRIGIN) return 0;
    const int n_split = m.n_osplit * m.n_ksplit;
    for (int q = 0; q < lv.n; ++q) {
        const int p = lv.order ? (int)((uint32_t)lv.order[q] & LV_POS_MASK) : q;
        const double *th = theta + (size_t)p * m.d;
        if (is_ssd(m.kind)) {
            for (int os = 0; os < m.n_osplit; ++os)
                for (int ks = 0; ks < m.n_ksplit; ++ks) {
                    const int k0 = ks * m.ksplit_len, k1 = std::min(m.ssd_k, k0 + m.ksplit_len);
                    const int64_t o0 = (int64_t)os * m.split_len, o1 = std::min<int64_t>(m.ssd_ld, o0 + m.split_len);
                    double s = 0.0;
                    for (int k = k0; k < k1; ++k) {
                        // DEMCMC_TEST_CORRUPT (mutation tests): the wrong dimension's mean, scaled and shifted
                        const double mean = m.debug_corrupt ? centred_mean(m, th, (k + 1) % m.ssd_k) * 3.0 + 17.0 : centred_mean(m, th, k);
                        for (int64_t i = o0; i < o1; ++i) s += m.xT[(int64_t)k * m.ssd_ld + i] * mean;
                    }
                    part[(size_t)p * n_split + os * m.n_ksplit + ks] = s;
                }
        } else {
            double par[MAX_ACC + 4];
            if (m.kind == M_GAUSSIAN) { par[0] = th[0]; par[1] = th[1]; par[2] = log(th[1]); }
            else if (m.kind == M_LNR) { for (int r = 0; r <= m.n_dim; ++r) par[r] = th[r]; }
            else {
                double pneg = 1.0;
                for (int r = 0; r < m.n_dim; ++r) { par[r] = th[r]; pneg *= norm_cdf(-th[r]); }
                par[m.n_dim] = th[m.n_dim]; par[m.n_dim + 1] = th[m.n_dim + 1]; par[m.n_dim + 2] = th[m.n_dim + 2];
                par[m.n_dim + 3] = 1.0 / (1.0 - pneg);
            }
            const double *sg = m.has_sigma ? m.sigma_acc : nullptr;
            for (int os = 0; os < m.n_osplit; ++os) {
                const int64_t i0 = (int64_t)os * m.split_len, i1 = std::min<int64_t>(m.n_obs, i0 + m.split_len);
                double s = 0.0;
                for (int64_t i = i0; i < i1; ++i) {
                    const int c = m.kind == M_GAUSSIAN ? 0 : m.choice[i] - 1;
                    if (m.kind == M_GAUSSIAN) s += gaussian_obs(par, m.x[i]);
                    else if (m.kind == M_LNR) s += lnr_obs(par, m.n_dim, sg, m.x[i], c);
                    else s += lba_obs(par, m.n_dim, par[m.n_dim + 3], m.lba_floor, m.x[i], c);
                }
                part[(size_t)p * n_split + os] = s;
            }
        }
    }
    return 0;
}

int launch_loglik(const ConfigDev &, const ModelDev &m, const double *theta, const Level &lv, double *part, long long *)
{
    if (loglik_impl(m, theta, lv, part)) return -1;
    if (is_ssd(m.kind)) {
        const int n_split = m.n_osplit * m.n_ksplit;
        for (int q = 0; q < lv.n; ++q) {
            const uint32_t e = (uint32_t)lv.order[q];
            const SweepCtx &ctx = lv.ctxs[e >> LV_SLOT_SHIFT];
            const int p = (int)(e & LV_POS_MASK);
            double s = 0.0;
            for (int c = 0; c < n_split; ++c) s += part[(size_t)p * n_split + c];
            ctx.ll_acc[p] = 1;
            ctx.ll_q[p] = s;
        }
    }
    return 0;
}

int launch_eval(const ConfigDev &cfg, const ModelDev &m, const double *theta, int64_t n, double *ll, double *prior, double *w, double *part, double *xdot)
{
    Level lv; lv.order = nullptr; lv.n = (int32_t)n; lv.ctxs = nullptr;
    loglik_impl(m, theta, lv, part);
    ++g_launches;
    const SerialLanes co;
    const int n_split = m.n_osplit * m.n_ksplit;
    for (int64_t i = 0; i < n; ++i) {
        const double *th = theta + (size_t)i * cfg.d;
        bool inb; double pr;
        bounds_and_prior(co, cfg, m, th, inb, pr);
        double s = 0.0;
        if (m.kind != M_BINOMIAL && m.kind != M_RASTRIGIN) for (int q = 0; q < n_split; ++q) s += part[(size_t)i * n_split + q];
        const double l = finalize_ll(m, th, s, mean_sq(co, m, th));
        if (ll) ll[i] = l;
        if (xdot) xdot[i] = s;
        if (prior) prior[i] = inb ? pr : -inf();
        if (w) w[i] = cfg.fitness == FITNESS_FUN ? (inb ? l : (cfg.update == UPDATE_MAXIMIZE ? -inf() : inf())) : (inb ? pr + l : -inf());
    }
    return 0;
}

int launch_base_prep(const ConfigDev &cfg, const double *w, double *th, double *cw, double *tot)
{
    ++g_launches;
    const int Np = cfg.Np;
    for (int g = 0; g < cfg.G_local; ++g) {
        const double *wg = w + (size_t)g * Np;
        double *tg = th + (size_t)g * Np, *cg = cw + (size_t)g * Np;
        ksum_t k = { 0, 0 };
        for (int i = 0; i < Np; ++i) { tg[i] = exp(wg[i]); kadd(k, tg[i]); }
        const double t = kval(k);
        bool bad = false;
        for (int i = 0; i < Np; ++i) { tg[i] = tg[i] / t; bad |= tg[i] != tg[i]; }
        const double *src = bad ? wg : tg;
        ksum_t k2 = { 0, 0 };
        for (int i = 0; i < Np; ++i) kadd(k2, src[i]);
        tot[g] = kval(k2);
        double c = src[0];
        cg[0] = c;
        for (int i = 1; i < Np; ++i) { c += src[i]; cg[i] = c; }
    }
    return 0;
}

int launch_plan(const ConfigDev &cfg, const SweepCtx *ctxs, int n_sw)
{
    ++g_launches;
    const int P = cfg.G_local * cfg.Np;
    for (int s = 0; s < n_sw; ++s)
        if (ctxs[s].plan)
            for (int p = 0; p < P; ++p) ctxs[s].plan[p] = make_plan(cfg, ctxs[s], p);
    return 0;
}

int launch_propose(const ConfigDev &cfg, const ModelDev &m, const Level &lv)
{
    ++g_launches;
    for (int q = 0; q < lv.n; ++q) {
        const uint32_t e = (uint32_t)lv.order[q];
        const SweepCtx &ctx = lv.ctxs[e >> LV_SLOT_SHIFT];
        const int p = (int)(e & LV_POS_MASK);
        NullSink sink;
        propose_particle(SerialLanes(), cfg, m, ctx, p, sink);
        ctx.prop_msq[p] = mean_sq(SerialLanes(), m, ctx.prop_theta + (size_t)p * cfg.d);
    }
    return 0;
}

// the persistent chunk kernel exists on the device only: the engine falls back to level-by-level launches
int launch_moments(const double *x, int64_t n, int32_t d, double *mean, double *m2)
{
    ++g_launches;
    for (int k = 0; k < d; ++k) {                                       // about the first vector, as the kernels
        double mu = 0.0, s = 0.0;
        for (int64_t r = 0; r < n; ++r) { const double v = x[r * d + k] - x[k], dl = v - mu; mu += dl / (double)(r + 1); s += dl * (v - mu); }
        mean[k] = x[k] + mu; m2[k] = s;
    }
    return 0;
}

int launch_diag_pos(const int32_t *rid, int64_t row0, int64_t n_rows, int32_t P, int32_t id_base, int32_t P_ids, int32_t pos_base, int32_t *pos)
{
    ++g_launches;
    for (int64_t r = 0; r < n_rows; ++r)
        for (int s = 0; s < P; ++s) { const int id = rid[(row0 + r) * P + s] - id_base; if (id >= 0 && id < P_ids) pos[(size_t)r * P_ids + id] = pos_base + s; }
    return 0;
}
int diag_max_half() { return 24576; }
int diag_max_lags() { return 4096; }
int launch_diag_aggregates(const DiagShards &sh, const int32_t *pos, int64_t row0, int64_t n_rows, int32_t P, int32_t d, int32_t lag0, int32_t n_lag, double *agg)
{
    ++g_launches;
    const int64_t nh = n_rows / 2;
    std::vector<double> x(nh);
    for (int k = 0; k < d; ++k) {
        double *a = agg + (size_t)k * (3 + n_lag);
        for (int j = 0; j < 3 + n_lag; ++j) a[j] = 0.0;
        const int q0 = pos[0], shard0 = q0 / sh.P_local;               // the kernel's shift: the draw of id 0 at row0
        const double shift = sh.theta[shard0][(row0 * sh.P_local + (q0 - shard0 * sh.P_local)) * d + k];
        for (int c = 0; c < 2 * P; ++c) {
            const int id = c >> 1;
            const int64_t r0 = (c & 1) ? n_rows - nh : 0;
            double mean = 0.0;
            for (int64_t i = 0; i < nh; ++i) {
                const int q = pos[(size_t)(r0 + i) * P + id], shard = q / sh.P_local;
                x[i] = sh.theta[shard][((row0 + r0 + i) * sh.P_local + (q - shard * sh.P_local)) * d + k] - shift;
                mean += x[i];
            }
            mean /= (double)nh;
            for (int64_t i = 0; i < nh; ++i) x[i] -= mean;
            for (int tl = 0; tl < n_lag; ++tl) {
                const int t = lag0 + tl;
                double s = 0.0;
                for (int64_t i = 0; i + t < nh; ++i) s += x[i] * x[i + t];
                s /= (double)nh;
                a[3 + tl] += s;
                if (t == 0) { a[0] += s * (double)nh / (double)(nh - 1); a[1] += mean; a[2] += mean * mean; }
            }
        }
    }
    return 0;
}

int launch_level_fused(const ConfigDev &, const ModelDev &, const Level &) { return 1; }
int launch_chunk_small(const ConfigDev &, const ModelDev &, const int32_t *, const SweepCtx *, const int32_t *, int) { return 1; }
int chunk_persist_lanes(const ConfigDev &, const ModelDev &) { return 0; }
int launch_chunk_persist(const ConfigDev &, const ModelDev &, const int32_t *, const SweepCtx *, const int32_t *, const int32_t *,
                         const int32_t *, int, int, long long *, int) { return 1; }

int launch_accept(const ConfigDev &cfg, const ModelDev &m, const Level &lv)
{
    ++g_launches;
    for (int q = 0; q < lv.n; ++q) {
        const uint32_t e = (uint32_t)lv.order[q];
        accept_particle(SerialLanes(), cfg, m, lv.ctxs[e >> LV_SLOT_SHIFT], (int)(e & LV_POS_MASK));
    }
    return 0;
}

static int select_particle(const double *w, int Np, double u)
{
    std::vector<double> th(Np);
    ksum_t k = { 0, 0 };
    for (int i = 0; i < Np; ++i) { th[i] = exp(-w[i]); kadd(k, th[i]); }
    const double tot = kval(k);
    bool bad = false;
    for (int i = 0; i < Np; ++i) { th[i] /= tot; bad |= th[i] != th[i]; }
    int r = 0;
    if (bad) { for (int i = 0; i < Np; ++i) { if (w[i] != w[i]) { r = i; break; } if (w[i] < w[r]) r = i; } return r; }
    ksum_t k2 = { 0, 0 };
    for (int i = 0; i < Np; ++i) kadd(k2, th[i]);
    const double t = u * kval(k2);
    double cw = th[0];
    while (cw < t && r < Np - 1) { ++r; cw += th[r]; }
    return r;
}

static int select_base(const double *w, int Np, double u)
{
    std::vector<double> th(Np);
    ksum_t k = { 0, 0 };
    for (int i = 0; i < Np; ++i) { th[i] = exp(w[i]); kadd(k, th[i]); }
    const double tot = kval(k);
    bool bad = false;
    for (int i = 0; i < Np; ++i) { th[i] /= tot; bad |= th[i] != th[i]; }
    const double *src = bad ? w : th.data();
    ksum_t k2 = { 0, 0 };
    for (int i = 0; i < Np; ++i) kadd(k2, src[i]);
    const double t = u * kval(k2);
    int r = 0;
    double cw = src[0];
    while (cw < t && r < Np - 1) { ++r; cw += src[r]; }
    return r;
}

int launch_mig_pick(const ConfigDev &cfg, const MigArgs &a, const double *w, int32_t *picks)
{
    ++g_launches;
    for (int i = 0; i < a.n; ++i) {
        const int gl = a.groups[i] - cfg.group_begin;
        picks[i] = (gl < 0 || gl >= cfg.G_local) ? -1 : select_particle(w + (size_t)gl * cfg.Np, cfg.Np, a.u_pick[i]);
    }
    return 0;
}

int launch_mig_gather(const ConfigDev &cfg, const MigArgs &a, const int32_t *picks, const double *theta, const double *w, const int32_t *id, const uint8_t *acc, double *stage)
{
    ++g_launches;
    for (int i = 0; i < a.n; ++i) {
        const int gl = a.groups[i] - cfg.group_begin;
        if (gl < 0 || gl >= cfg.G_local) continue;
        const size_t p = (size_t)gl * cfg.Np + picks[i];
        double *row = stage + (size_t)i * (cfg.d + 3);
        memcpy(row, theta + p * cfg.d, sizeof(double) * cfg.d);
        row[cfg.d] = w[p]; row[cfg.d + 1] = (double)id[p]; row[cfg.d + 2] = (double)acc[p];
    }
    return 0;
}

// The migration mailbox of the double: host memory shared by the threads of one process (a multi-device handle runs
// one thread per "device"); same protocol as k_mig_push / k_mig_scatter -- rows, then a release store of the tag.
int launch_mig_scatter(const ConfigDev &cfg, const MigArgs &a, const int32_t *picks, const double *stage, double *theta, double *w, int32_t *id, uint8_t *acc, int32_t *pos,
                       const Mbox *mbox, int rank, int slot, unsigned long long tag)
{
    ++g_launches;
    for (int i = 0; i < a.n; ++i) {
        const int gl = a.groups[i] - cfg.group_begin;
        if (gl < 0 || gl >= cfg.G_local) continue;
        const size_t p = (size_t)gl * cfg.Np + picks[i];
        const int r = (i + a.n - 1) % a.n;
        const double *row = stage + (size_t)r * (cfg.d + 3);
        if (mbox && mbox->rows && a.src_rank[i] != rank) {
            const size_t cell = (size_t)slot * mbox->max_rows + r;
            while (__atomic_load_n(mbox->flags + cell, __ATOMIC_ACQUIRE) != tag) sched_yield();
            row = mbox->rows + cell * mbox->row_len;
        }
        memcpy(theta + p * cfg.d, row, sizeof(double) * cfg.d);
        w[p] = row[cfg.d]; id[p] = (int32_t)row[cfg.d + 1]; acc[p] = (uint8_t)row[cfg.d + 2];
        if (pos) pos[id[p] - cfg.group_begin * cfg.Np] = (int32_t)p;
    }
    return 0;
}

int launch_history_by_id(const double *rt, const double *rw, const uint8_t *ra, const int32_t *rid, int64_t n_rows_dev, int64_t row0,
                         int64_t n_rows_out, int32_t P, int32_t d, int32_t id_base, double *samples, double *lp, uint8_t *accept, int32_t P_ids)
{
    ++g_launches;
    if (P_ids <= 0) P_ids = P;
    for (int64_t r = 0; r < n_rows_dev; ++r)
        for (int slot = 0; slot < P; ++slot) {
            const int id = rid[r * P + slot] - id_base;
            if (id < 0 || id >= P_ids) continue;
            const int64_t ro = row0 + r;
            if (samples) for (int k = 0; k < d; ++k) samples[((int64_t)id * d + k) * n_rows_out + ro] = rt[(r * P + slot) * d + k];
            if (lp) lp[(int64_t)id * n_rows_out + ro] = rw[r * P + slot];
            if (accept) accept[(int64_t)id * n_rows_out + ro] = ra[r * P + slot];
        }
    return 0;
}

int launch_chains(const double *rt, const double *rw, const uint8_t *ra, const int32_t *rid, const int32_t *final_id, int32_t *pos,
                  int64_t row0, int64_t n_rows, int32_t P, int32_t d, int32_t id_base, double *out, int32_t P_ids, int32_t pos_base, int phase)
{
    ++g_launches;
    if (P_ids <= 0) P_ids = P;
    if (phase & 1) for (int c = 0; c < P; ++c) { const int id = final_id[c] - id_base; if (id >= 0 && id < P_ids) pos[id] = pos_base + c; }
    if (!(phase & 2)) return 0;
    for (int64_t r = 0; r < n_rows; ++r)
        for (int slot = 0; slot < P; ++slot) {
            const int64_t row = row0 + r;
            const int id = rid[row * P + slot] - id_base;
            if (id < 0 || id >= P_ids) continue;
            for (int k = 0; k < d; ++k) out[((int64_t)id * (d + 2) + k) * n_rows + r] = rt[(row * P + slot) * d + k];
            out[((int64_t)pos[id] * (d + 2) + d) * n_rows + r] = (double)ra[row * P + slot];
            out[((int64_t)pos[id] * (d + 2) + d + 1) * n_rows + r] = rw[row * P + slot];
        }
    return 0;
}

int launch_op_project(const double *p1, const double *p2, int d, double *out)
{
    double v1 = 0, v2 = 0;
    for (int k = 0; k < d; ++k) { v1 += p1[k] * p2[k]; v2 += p2[k] * p2[k]; }
    for (int k = 0; k < d; ++k) out[k] = p2[k] * (v1 / v2);
    return 0;
}
int launch_op_snooker(const double *pt, const double *pz, const double *pm, const double *pn, double g, const double *b, int d, double *out, double *log_adj)
{
    double v1m = 0, v1n = 0, v2 = 0;
    for (int k = 0; k < d; ++k) { const double pd = pt[k] - pz[k]; v1m += pm[k] * pd; v1n += pn[k] * pd; v2 += pd * pd; }
    double sq1 = 0, sq2 = 0;
    for (int k = 0; k < d; ++k) {
        out[k] = snooker_elem(pt[k], pz[k], v1m / v2, v1n / v2, g, b[k]);
        sq1 += (out[k] - pz[k]) * (out[k] - pz[k]); sq2 += (pt[k] - pz[k]) * (pt[k] - pz[k]);
    }
    *log_adj = adjust_loglike(sq1, sq2, d);
    return 0;
}
int launch_op_de(const double *pt, const double *pm, const double *pn, const double *pb, double g1, double g2, const double *b, int d, double *out)
{
    for (int k = 0; k < d; ++k) out[k] = de_elem(pt[k], pm[k], pn[k], pb ? pb[k] : pt[k], g1, g2, pb != nullptr, b[k]);
    return 0;
}
int launch_op_reset(const double *prop, const double *pt, const uint8_t *mask, int d, double *out)
{
    for (int k = 0; k < d; ++k) out[k] = mask[k] ? prop[k] : pt[k];
    return 0;
}
int launch_op_accept(const double *wp, const double *wc, const double *adj, const double *u, int n, uint8_t *out)
{
    for (int i = 0; i < n; ++i) out[i] = accept(wp[i], wc[i], adj[i], u[i]) ? 1 : 0;
    return 0;
}
int launch_op_select(const double *w, int n, double u, int32_t *base_idx, int32_t *mig_idx)
{
    *base_idx = select_base(w, n, u);
    *mig_idx = select_particle(w, n, u);
    return 0;
}
int fp64_peak(double *t) { *t = 0.0; return 0; }
int fp64_peaks(double *a, double *b) { if (a) *a = 0.0; if (b) *b = 0.0; return 0; }
int copy_peak(double *g) { *g = 0.0; return 0; }

int launch_mig_push(const ConfigDev &cfg, const MigArgs &a, const double *stage, const PeerTable &peers, const Mbox &geom, int rank, int slot, unsigned long long tag)
{
    ++g_launches;
    for (int i = 0; i < a.n; ++i) {
        if (a.src_rank[i] != rank || a.dst_rank[i] == rank) continue;
        const int r = (i + a.n - 1) % a.n, dst = a.dst_rank[i];
        const size_t cell = (size_t)slot * geom.max_rows + r;
        memcpy(peers.rows[dst] + cell * geom.row_len, stage + (size_t)r * (cfg.d + 3), sizeof(double) * (cfg.d + 3));
        __atomic_store_n(peers.flags[dst] + cell, tag, __ATOMIC_RELEASE);
    }
    return 0;
}
int mbox_create(int depth, int max_rows, int row_len, Mbox *out)
{
    out->depth = depth; out->max_rows = max_rows; out->row_len = row_len;
    out->rows = (double *)calloc((size_t)depth * max_rows * row_len, sizeof(double));
    out->flags = (unsigned long long *)calloc((size_t)depth * max_rows, sizeof(unsigned long long));
    return (out->rows && out->flags) ? 0 : -1;
}
void mbox_destroy(Mbox *m) { free(m->rows); free(m->flags); m->rows = nullptr; m->flags = nullptr; }
int mbox_export(const Mbox &, uint8_t *) { g_err = "the test double has no inter-process mailbox"; return -1; }
int mbox_open(const uint8_t *, Mbox *) { g_err = "the test double has no inter-process mailbox"; return -1; }
void mbox_close(Mbox *) {}
int enable_peer_access(int, int) { return 0; }
int comm_barrier(void *) { return 0; }
int comm_unique_id(uint8_t id[128]) { memset(id, 0, 128); return 0; }
int comm_init(const uint8_t *, int, int, void **comm) { *comm = malloc(8); return 0; }
int comm_destroy(void *comm) { free(comm); return 0; }
typedef int (*allgather_fn)(const void *send, void *recv, size_t bytes_per_rank, void *user);
static allgather_fn g_allgather = nullptr;
static void *g_allgather_user = nullptr;
int comm_allgather(void *, const void *send, void *recv, size_t bytes_per_rank)
{
    if (!g_allgather) { g_err = "emu: no allgather hook installed"; return -1; }
    return g_allgather(send, recv, bytes_per_rank, g_allgather_user);
}
int launch_pos_from_ids(const int32_t *ids, int32_t n, int32_t *pos)
{
    ++g_launches;
    for (int q = 0; q < n; ++q) if (ids[q] >= 0 && ids[q] < n) pos[ids[q]] = q;
    return 0;
}
int comm_exchange(void *, int rank, int n, const int *src_rank, const int *dst_rank, double *send, double *recv, int row_len)
{
    if (!g_exchange) { g_err = "emu: no exchange hook installed"; return -1; }
    return g_exchange(rank, n, src_rank, dst_rank, send, recv, row_len, g_exchange_user);
}

} // namespace be
} // namespace de

extern "C" void demcmc_emu_set_allgather(de::be::allgather_fn fn, void *user)
{
    de::be::g_allgather = fn;
    de::be::g_allgather_user = user;
}
extern "C" void demcmc_emu_set_exchange(de::be::exchange_fn fn, void *user)
{
    de::be::g_exchange = fn;
    de::be::g_exchange_user = user;
}

// ---- property check of the planner (tests/test_planner_properties.py): every update of a chunk appears
// exactly once, and every dependency of an update -- its own previous update, donors with a smaller slot in
// the same sweep, donors with a larger slot in the previous sweep (crossover.jl:12-17) -- sits in a strictly
// earlier level, with or without the octet shaping.  Returns 0, or a negative code naming the violation.
#include "planner.h"
extern "C" int demcmc_emu_plan_check_cap(uint64_t seed, int Np, int G, int n_sweeps, double beta, double theta_snooker, int shape,
                                          int sweep_stride, int cap, int *n_levels_out, int *padded_out);
extern "C" int demcmc_emu_plan_check(uint64_t seed, int Np, int G, int n_sweeps, double beta, double theta_snooker, int shape,
                                      int sweep_stride, int *n_levels_out, int *padded_out)
{
    return demcmc_emu_plan_check_cap(seed, Np, G, n_sweeps, beta, theta_snooker, shape, sweep_stride, 0, n_levels_out, padded_out);
}
// ... with a level capacity (PlanInput::level_cap): also checks that no level exceeds it; *padded_out = the largest level
extern "C" int demcmc_emu_plan_check_cap(uint64_t seed, int Np, int G, int n_sweeps, double beta, double theta_snooker, int shape,
                                          int sweep_stride, int cap, int *n_levels_out, int *padded_out)
{
    using namespace de;
    PlanInput in{};
    in.seed = seed; in.Np = Np; in.G_local = G; in.group_begin = 0; in.G_total = G; in.proposal = 0; in.beta = beta;
    in.theta_snooker = theta_snooker; in.resample = false; in.t_kind = nullptr; in.t_idx = nullptr; in.shape_octets = shape;
    in.sweep_stride = sweep_stride;
    in.level_cap = cap;
    bool bd[MAX_CHUNK] = { false };
    ChunkPlan pl;
    const uint32_t sweep0 = 7;
    plan_chunk(in, sweep0, n_sweeps, bd, pl);
    const int P = Np * G;
    std::vector<int> level((size_t)n_sweeps * P, -1);
    if ((int)pl.order.size() != n_sweeps * P || (int)pl.level_off.size() != pl.n_levels + 1) return -1;
    int padded = 0;
    for (int l = 0; l < pl.n_levels; ++l) {
        const int n = pl.level_off[l + 1] - pl.level_off[l];
        if (n < 0) return -2;
        if (cap > 0 && n > cap + (shape > 0 ? shape : 0)) return -7;       // (the octet shaping may hand a remainder of < shape updates down)
        padded += (n + 7) / 8 * 8;
        for (int q = pl.level_off[l]; q < pl.level_off[l + 1]; ++q) {
            const uint32_t e = (uint32_t)pl.order[q];
            const int s = (int)(e >> ENTRY_SLOT_SHIFT), p = (int)(e & ENTRY_POS_MASK);
            if (s < 0 || s >= n_sweeps || p < 0 || p >= P || level[(size_t)s * P + p] >= 0) return -3;
            level[(size_t)s * P + p] = l;
        }
    }
    for (int s = 0; s < n_sweeps; ++s)
        for (int g = 0; g < G; ++g) {
            const uint32_t sweep = sweep0 + (uint32_t)s * (uint32_t)sweep_stride;
            const bool mutate = pl.mutate[(size_t)s * G + g] != 0;
            if (mutate != (uniform2(seed, ST_MUT, sweep, (uint32_t)g, 0).a <= beta)) return -4;
            for (int j = 0; j < Np; ++j) {
                const int me = level[(size_t)s * P + g * Np + j];
                if (me < 0) return -5;
                if (s > 0 && level[(size_t)(s - 1) * P + g * Np + j] >= me) return -6;
                if (mutate) continue;
                const Plan pp = plan_particle(seed, sweep, (uint32_t)(g * Np + j), j, Np, false, theta_snooker);
                const int dep[3] = { pp.kind == KIND_SNOOKER ? pp.i0 : -1, pp.i1, pp.i2 };
                for (int q = 0; q < 3; ++q) {
                    const int k = dep[q];
                    if (k < 0 || k == j) continue;
                    if (k < j) { if (level[(size_t)s * P + g * Np + k] >= me) return -7; }
                    else if (s > 0 && level[(size_t)(s - 1) * P + g * Np + k] >= me) return -8;
                }
            }
        }
    if (n_levels_out) *n_levels_out = pl.n_levels;
    if (padded_out) *padded_out = padded;
    return 0;
}

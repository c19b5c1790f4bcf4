// engine.cpp -- host side of libdemcmc_b200: the handle, the iteration loop of _sample
// (src/main.jl:33-38) and the C ABI of include/demcmc_b200.h.  All arithmetic on particles happens
// in the kernels behind backend.h; the host only schedules (planner.h) and moves buffers.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <type_traits>
#include <array>
#include <vector>

#include "../../include/demcmc_b200.h"
#include "backend.h"
#include "de_types.h"
#include "planner.h"

using namespace de;

static thread_local std::string g_err;

static int fail(int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
#define BE(call) do { if ((call) != 0) return fail(DEMCMC_ECUDA, "%s: %s", #call, be::last_error()); } while (0)

namespace {

struct Row { double *theta; double *w; int32_t *id; uint8_t *acc; };

struct Upload {            // pinned staging + device copy of one sweep's schedule
    // ONE pinned block and ONE device block per slot, copied with one cudaMemcpyAsync per chunk:
    // [SweepCtx x MAX_CHUNK][mutate flags MAX_CHUNK x G, padded][level-sorted entries MAX_CHUNK x P]
    uint8_t *h_blk = nullptr, *d_blk = nullptr;
    size_t off_mut = 0, off_order = 0, bytes = 0;
    int32_t *h_order = nullptr, *d_order = nullptr;   // [MAX_CHUNK][P] level-sorted entries
    uint8_t *h_mut = nullptr, *d_mut = nullptr;       // [MAX_CHUNK][G]
    SweepCtx *h_ctx = nullptr, *d_ctx = nullptr;      // [MAX_CHUNK]
    void *copied = nullptr;  // event: the H2D copies out of the pinned buffers have run
    bool armed = false;
};

} // namespace

struct MultiState;
struct demcmc_handle {
    demcmc_config cfg;
    std::vector<uint8_t> blocks;
    std::vector<double> lo, hi;
    int G_local = 0, P = 0, B = 1, d = 0;
    ConfigDev dcfg;
    ModelDev dmodel;
    bool has_model = false, has_state = false;
    std::vector<void *> model_allocs;
    void *custom_mod = nullptr;                         // DEMCMC_CUSTOM: the likelihood module loaded on this device
    // state rows
    int64_t hist_cap = 0, iters_done = 0;
    int64_t iter_offset = 0;                            // iterations the chain ran before this handle (demcmc_set_iteration)
    std::vector<uint8_t> block_on;                      // blocking_on(de) per absolute iteration (demcmc_set_blocking_schedule); beyond it: on
    double *hist_theta = nullptr, *hist_w = nullptr;
    int32_t *hist_id = nullptr;
    uint8_t *hist_acc = nullptr;
    int32_t *hist_pos = nullptr;                        // resample: [row][id] -> position holding that id
    // resample on a sharded job: every rank keeps a replicated copy of every history row of ALL ranks
    // (positions in rank order) and its id -> global position map, gathered after each iteration
    double *ghist_theta = nullptr;                      // [row][P_total][d]
    int32_t *ghist_pos = nullptr;                       // [row][P_total]
    int32_t *gid_tmp = nullptr;                         // [2][P_total] gathered ids of one row (two copies: a multi-device handle alternates them)
    uint64_t n_gathers = 0;
    int64_t k_store = 1;                                // store_every: iteration it (1-based, counted on this handle) is kept iff it % k_store == 0
    int n_scratch = 3;                                  // scratch state rows (write-once within a chunk): 3, or MAX_CHUNK + 2 when thinning
    int64_t n0 = 0;                                     // de.n_initial: history rows before iteration 1
    bool has_history = false;                           // the n_initial prior rows were uploaded
    double *scr_theta = nullptr, *scr_w = nullptr;      // 3 scratch rows
    int32_t *scr_id = nullptr;
    uint8_t *scr_acc = nullptr;
    int scr_cursor = 0;                                 // last scratch row handed out (ring)
    int cur_scratch = 0;                                // current state lives in scratch row k, or
    int64_t cur_hist = -1;                              // in history row cur_hist (>= 0)
    // proposal scratch
    double *prop_theta = nullptr, *prop_prior = nullptr, *prop_adj = nullptr, *prop_msq = nullptr, *ll_part = nullptr, *ll_q = nullptr;
    PlanRec *plan_recs = nullptr;                      // [MAX_CHUNK][P_local] the pre-drawn plans of the chunk in flight (native mode)
    long long *ll_acc = nullptr;
    uint8_t *prop_inb = nullptr;
    double *base_th = nullptr, *base_cw = nullptr, *base_tot = nullptr;
    double *d_lo = nullptr, *d_hi = nullptr;
    uint8_t *d_blocks = nullptr;
    // schedule ring
    static constexpr int RING = 4;
    int max_chunk = MAX_CHUNK;                          // sweeps overlapped on the device (1 = a barrier per sweep)
    int n_lanes = 1;                                    // concurrent kernel chains over independent sets of groups (demcmc_set_lanes)
    Upload ring[RING];
    int64_t ring_use = 0;
    // migration
    int32_t *d_picks = nullptr;
    double *d_stage = nullptr, *d_stage_recv = nullptr;
    std::vector<int32_t> last_mig_slots;                // [n_iter][G_total] of the last call
    int32_t *d_mig_log = nullptr;                       // device log of picks of the last call
    int64_t mig_log_iters = 0;
    // trace of the last call
    double *tr_theta = nullptr, *tr_w = nullptr, *tr_adj = nullptr, *tr_xdot = nullptr;
    uint8_t *tr_acc = nullptr;
    int64_t tr_sweeps = 0;
    // comm
    void *comm = nullptr;
    int rank = 0, n_ranks = 1;
    // P2P migration mailbox (de_types.h: Mbox): this rank's own, and every rank's as mapped here.  Used instead of the
    // NCCL send/recv exchange when every peer could be mapped (multi-process: CUDA IPC; one process: peer access).
    Mbox mbox = { nullptr, nullptr, 0, 0, 0 };
    PeerTable peers = {};
    std::vector<Mbox> peer_maps;                        // IPC mappings to close (multi-process)
    bool mbox_on = false;
    bool mbox_shared = false;                           // the mailbox belongs to the process-wide cache (multi-process jobs)
    uint64_t mbox_seq = 0, *mbox_seq_p = &mbox_seq;     // cross-rank migration events so far (the same on every rank)
    std::function<int()> mbox_barrier;                  // all ranks have consumed every event so far (slot reuse)
    // multi-device handle (cfg.n_devices > 1): one child handle per device, driven by one host thread each
    std::vector<demcmc_handle *> kids;
    demcmc_handle *parent = nullptr;
    struct MultiState *multi = nullptr;
    std::vector<int32_t> devices;
    std::vector<int> group_owner;                       // [G_total] rank owning each group
    demcmc_counters ctr;
    // measurement mode (demcmc_set_timing)
    int64_t flush_bytes = 0;
    bool time_loglik = false;
    bool suffstat = false;                              // demcmc_set_sufficient_stat: the O(N d) stream is skipped
    void *flush_buf = nullptr;
    std::vector<void *> tev;                            // pool of timing events
};

static Row row_of(demcmc_handle *h, bool hist, int64_t idx)
{
    const size_t P = h->P, d = h->d;
    Row r;
    if (hist) { r.theta = h->hist_theta + idx * P * d; r.w = h->hist_w + idx * P; r.id = h->hist_id + idx * P; r.acc = h->hist_acc + idx * P; }
    else { r.theta = h->scr_theta + idx * P * d; r.w = h->scr_w + idx * P; r.id = h->scr_id + idx * P; r.acc = h->scr_acc + idx * P; }
    return r;
}
// history rows held after `iters` iterations of this handle: the n_initial prior rows + every k_store-th iteration
static int64_t stored_rows(const demcmc_handle *h, int64_t iters) { return h->n0 + iters / h->k_store; }
static int64_t stored_rows(const demcmc_handle *h) { return stored_rows(h, h->iters_done); }
static Row cur_row(demcmc_handle *h) { return h->cur_hist >= 0 ? row_of(h, true, h->cur_hist) : row_of(h, false, h->cur_scratch); }

// history rows: [0, n0) = the n_initial prior rows (utilities.jl:35-39), row n0 + it = iteration it
static int grow_history(demcmc_handle *h, int64_t need)
{
    if (need <= h->hist_cap) return 0;
    // exactly what the call needs the first time (sample() runs once: no over-allocation); a handle that keeps
    // being extended grows by halves so the copies stay amortised
    int64_t cap = h->hist_cap > 0 ? std::max<int64_t>(need, h->hist_cap + h->hist_cap / 2) : need;
    const size_t P = h->P, d = h->d;
    const int64_t have = h->hist_cap > 0 ? stored_rows(h) : 0;
    double *nt = (double *)be::dmalloc(sizeof(double) * cap * P * d);
    double *nw = (double *)be::dmalloc(sizeof(double) * cap * P);
    int32_t *ni = (int32_t *)be::dmalloc(sizeof(int32_t) * cap * P);
    uint8_t *na = (uint8_t *)be::dmalloc(cap * P);
    int32_t *np = h->cfg.donors ? (int32_t *)be::dmalloc(sizeof(int32_t) * cap * P) : nullptr;
    if (!nt || !nw || !ni || !na || (h->cfg.donors && !np)) return fail(DEMCMC_ENOMEM, "history of %lld rows does not fit on the device", (long long)cap);
    if (have > 0) {
        BE(be::d2d(nt, h->hist_theta, sizeof(double) * have * P * d));
        BE(be::d2d(nw, h->hist_w, sizeof(double) * have * P));
        BE(be::d2d(ni, h->hist_id, sizeof(int32_t) * have * P));
        BE(be::d2d(na, h->hist_acc, have * P));
        if (np) BE(be::d2d(np, h->hist_pos, sizeof(int32_t) * have * P));
        BE(be::sync());
    }
    if (h->cfg.donors && h->n_ranks > 1) {
        const size_t Pt = (size_t)h->cfg.n_groups * h->cfg.Np;
        double *gt = (double *)be::dmalloc(sizeof(double) * cap * Pt * d);
        int32_t *gp = (int32_t *)be::dmalloc(sizeof(int32_t) * cap * Pt);
        if (!h->gid_tmp) h->gid_tmp = (int32_t *)be::dmalloc(sizeof(int32_t) * 2 * Pt);
        if (!gt || !gp || !h->gid_tmp) return fail(DEMCMC_ENOMEM, "replicated history of %lld rows does not fit on the device", (long long)cap);
        if (have > 0 && h->ghist_theta) {
            BE(be::d2d(gt, h->ghist_theta, sizeof(double) * have * Pt * d));
            BE(be::d2d(gp, h->ghist_pos, sizeof(int32_t) * have * Pt));
            BE(be::sync());
        }
        be::dfree(h->ghist_theta); be::dfree(h->ghist_pos);
        h->ghist_theta = gt; h->ghist_pos = gp;
    }
    be::dfree(h->hist_theta); be::dfree(h->hist_w); be::dfree(h->hist_id); be::dfree(h->hist_acc); be::dfree(h->hist_pos);
    h->hist_theta = nt; h->hist_w = nw; h->hist_id = ni; h->hist_acc = na; h->hist_pos = np; h->hist_cap = cap;
    return 0;
}

// resample on a sharded job: the replicated copy of history row `row` (theta and the id -> position
// map) from every rank's slice, in rank order = global position order
static int gather_row_local(demcmc_handle *h, int64_t row);
static int gather_row(demcmc_handle *h, int64_t row)
{
    if (h->parent) return gather_row_local(h, row);
    const size_t P = h->P, d = h->d, Pt = (size_t)h->cfg.n_groups * h->cfg.Np;
    if (be::comm_allgather(h->comm, h->hist_theta + (size_t)row * P * d, h->ghist_theta + (size_t)row * Pt * d, sizeof(double) * P * d) ||
        be::comm_allgather(h->comm, h->hist_id + (size_t)row * P, h->gid_tmp, sizeof(int32_t) * P) ||
        be::launch_pos_from_ids(h->gid_tmp, (int32_t)Pt, h->ghist_pos + (size_t)row * Pt))
        return fail(DEMCMC_ECOMM, "history gather: %s", be::last_error());
    return 0;
}

// ---- particle algebra ops (known-answer tests) --------------------------------------------------
namespace {
struct DevBuf {
    std::vector<void *> p;
    ~DevBuf() { for (void *q : p) be::dfree(q); }
    template <typename T> T *up(const T *src, size_t n)
    {
        T *q = (T *)be::dmalloc(std::max<size_t>(8, sizeof(T) * n));
        if (!q) return nullptr;
        p.push_back(q);
        if (src && n && be::h2d(q, src, sizeof(T) * n)) return nullptr;
        return q;
    }
};
int op_begin(int device)
{
    if (be::device_count() <= 0) return fail(DEMCMC_ENODEVICE, "no CUDA device: libdemcmc_b200 has no CPU fallback");
    if (be::set_device(device)) return fail(DEMCMC_ENODEVICE, "cannot select device %d", device);
    return 0;
}
} // namespace

// ---- P2P migration mailbox ------------------------------------------------------------------------------------
static bool mbox_wanted()
{
    const char *e = getenv("DEMCMC_MIG");                 // DEMCMC_MIG=nccl: keep the NCCL send/recv exchange (A/B runs, fallback)
    return !(e && strcmp(e, "nccl") == 0);
}
// Multi-process jobs keep ONE mailbox (and its IPC mappings of every peer) per device for the life of the process,
// like the NCCL communicator: handles come and go (one per sample() call), the mapping does not, so nothing exported
// is ever freed under a peer and a new handle pays no IPC set-up.  The event counter lives with the mailbox and only
// ever grows, so a flag left by an earlier handle can never equal a later tag.
struct MboxShared { size_t cap_doubles = 0, cap_flags = 0; int n_ranks = 0, rank = -1; Mbox box = { nullptr, nullptr, 0, 0, 0 }; PeerTable peers = {}; uint64_t seq = 0; };
static MboxShared g_mbox_shared[64];
static void mbox_geometry(const demcmc_handle *h, int *depth, int *max_rows, int *row_len)
{
    *row_len = h->d + 3; *max_rows = std::min(h->cfg.n_groups, (int)MAX_MIG);
    const size_t ev_bytes = sizeof(double) * (size_t)*row_len * *max_rows;
    *depth = (int)std::max<size_t>(16, std::min<size_t>(1024, ((size_t)64 << 20) / std::max<size_t>(1, ev_bytes)));
}
static int mbox_alloc(demcmc_handle *h)
{
    const int row_len = h->d + 3, max_rows = std::min(h->cfg.n_groups, (int)MAX_MIG);
    const size_t ev_bytes = sizeof(double) * (size_t)row_len * max_rows;
    const int depth = (int)std::max<size_t>(16, std::min<size_t>(1024, ((size_t)64 << 20) / std::max<size_t>(1, ev_bytes)));
    if (be::mbox_create(depth, max_rows, row_len, &h->mbox)) return -1;
    return 0;
}

// ---- multi-device handle: fan a call out over the children, one host thread per device -------------------------
namespace {
struct HostBarrier {
    std::mutex m; std::condition_variable cv; int n = 0, waiting = 0; uint64_t gen = 0; bool aborted = false;
    // false: a peer thread has left its run with an error (abort()) -- nobody would ever complete this barrier
    bool wait()
    {
        std::unique_lock<std::mutex> lk(m);
        if (aborted) return false;
        const uint64_t g = gen;
        if (++waiting == n) { waiting = 0; ++gen; cv.notify_all(); return true; }
        cv.wait(lk, [&] { return gen != g || aborted; });
        return gen != g;
    }
    void abort() { std::lock_guard<std::mutex> lk(m); aborted = true; cv.notify_all(); }
    void reset() { std::lock_guard<std::mutex> lk(m); aborted = false; waiting = 0; }
};
}
struct MultiState { HostBarrier barrier; };

// the same gather between the devices of a multi-device handle (one host thread per device, peer access enabled by
// multi_create): every device stores its slice of the row into every device's replicated copy, then all meet at a host
// barrier.  The gathered ids alternate between two buffers: a device may start the stores of gather n + 1 while a slower
// peer's position kernel of gather n is still queued; it cannot reach gather n + 2 before that peer has synchronised.
static int gather_row_local(demcmc_handle *h, int64_t row)
{
    demcmc_handle *p = h->parent;
    const size_t P = h->P, d = h->d, Pt = (size_t)h->cfg.n_groups * h->cfg.Np, par = (size_t)(h->n_gathers++ & 1);
    for (demcmc_handle *k : p->kids) {
        if (!k->ghist_theta || !k->gid_tmp) return fail(DEMCMC_ESTATE, "history gather: device %d has no replicated history", k->cfg.device);
        if (be::d2d(k->ghist_theta + ((size_t)row * Pt + (size_t)h->rank * P) * d, h->hist_theta + (size_t)row * P * d, sizeof(double) * P * d) ||
            be::d2d(k->gid_tmp + par * Pt + (size_t)h->rank * P, h->hist_id + (size_t)row * P, sizeof(int32_t) * P))
            return fail(DEMCMC_ECOMM, "history gather: %s", be::last_error());
    }
    if (be::sync()) return fail(DEMCMC_ECOMM, "history gather: %s", be::last_error());
    if (!p->multi->barrier.wait()) return fail(DEMCMC_ECOMM, "history gather: another device of the handle failed");
    if (be::launch_pos_from_ids(h->gid_tmp + par * Pt, (int32_t)Pt, h->ghist_pos + (size_t)row * Pt)) return fail(DEMCMC_ECOMM, "history gather: %s", be::last_error());
    return 0;
}

template <class F>
static int for_kids(demcmc_handle *h, F f, bool parallel = true)
{
    const size_t n = h->kids.size();
    std::vector<int> rc(n, 0);
    std::vector<std::string> msg(n);
    if (!parallel || n == 1) {
        for (size_t i = 0; i < n; ++i) { rc[i] = f(h->kids[i], (int)i); if (rc[i]) { msg[i] = g_err; break; } }
    } else {
        std::vector<std::thread> th;
        for (size_t i = 0; i < n; ++i)
            th.emplace_back([&, i]() { rc[i] = f(h->kids[i], (int)i); if (rc[i]) msg[i] = g_err; });     // g_err is thread-local
        for (auto &t : th) t.join();
    }
    for (size_t i = 0; i < n; ++i) if (rc[i]) return fail(rc[i], "device %d: %s", h->kids[i]->cfg.device, msg[i].c_str());
    return 0;
}


// ---- the multi-device entry points (cfg.n_devices > 1) ---------------------------------------------------------
static int multi_create(const demcmc_config *cfg, demcmc_handle **out)
{
    const int N = cfg->n_devices;
    if (!cfg->devices) return fail(DEMCMC_EINVAL, "n_devices = %d but devices is NULL", N);
    if (N > MAX_RANKS) return fail(DEMCMC_EUNSUPPORTED, "n_devices > %d", (int)MAX_RANKS);
    if (cfg->n_groups % N) return fail(DEMCMC_EINVAL, "n_groups %d is not a multiple of the %d devices", cfg->n_groups, N);
    if (cfg->group_begin != 0 || (cfg->group_count != 0 && cfg->group_count != cfg->n_groups)) return fail(DEMCMC_EINVAL, "a multi-device handle holds every group: group_begin / group_count must be 0");
    for (int i = 0; i < N; ++i) for (int j = 0; j < i; ++j) if (cfg->devices[i] == cfg->devices[j]) return fail(DEMCMC_EINVAL, "device %d listed twice", cfg->devices[i]);
    if (be::device_count() <= 0) return fail(DEMCMC_ENODEVICE, "no CUDA device: libdemcmc_b200 has no CPU fallback (%s)", be::last_error());
    demcmc_handle *p = new demcmc_handle();
    p->cfg = *cfg; p->cfg.devices = nullptr;
    p->devices.assign(cfg->devices, cfg->devices + N);
    p->d = cfg->d; p->n0 = cfg->n_initial; p->k_store = std::max(1, cfg->store_every);
    p->G_local = cfg->n_groups; p->P = cfg->n_groups * cfg->Np; p->B = cfg->n_blocks > 0 ? cfg->n_blocks : 1;
    memset(&p->ctr, 0, sizeof p->ctr);
    p->multi = new MultiState();
    p->multi->barrier.n = N;
    const int per = cfg->n_groups / N;
    for (int i = 0; i < N; ++i) {
        demcmc_config c = *cfg;
        c.n_devices = 0; c.devices = nullptr; c.device = cfg->devices[i]; c.group_begin = i * per; c.group_count = per;
        demcmc_handle *k = nullptr;
        const int rc = demcmc_create(&c, &k);
        if (rc) { const std::string m = g_err; demcmc_destroy(p); return fail(rc, "device %d: %s", c.device, m.c_str()); }
        k->parent = p; k->rank = i; k->n_ranks = N;
        for (int g = 0; g < cfg->n_groups; ++g) k->group_owner[g] = g / per;
        p->kids.push_back(k);
    }
    // migration between the devices: peer-mapped mailboxes, no host call between a device's chunks
    for (int i = 0; i < N; ++i) {
        demcmc_handle *k = p->kids[i];
        if (be::set_device(k->cfg.device) || mbox_alloc(k)) { const std::string m = be::last_error(); demcmc_destroy(p); return fail(DEMCMC_ENOMEM, "migration mailbox on device %d: %s", cfg->devices[i], m.c_str()); }
        for (int j = 0; j < N; ++j)
            if (j != i && be::enable_peer_access(cfg->devices[i], cfg->devices[j])) {
                const std::string m = be::last_error(); demcmc_destroy(p);
                return fail(DEMCMC_EUNSUPPORTED, "devices %d and %d: %s (a multi-device handle needs P2P between its GPUs; shard over processes with demcmc_comm_init otherwise)", cfg->devices[i], cfg->devices[j], m.c_str());
            }
    }
    for (int i = 0; i < N; ++i) {
        demcmc_handle *k = p->kids[i];
        for (int j = 0; j < N; ++j) { k->peers.rows[j] = p->kids[j]->mbox.rows; k->peers.flags[j] = p->kids[j]->mbox.flags; }
        k->mbox_on = true;
        MultiState *ms = p->multi;
        k->mbox_barrier = [ms]() { if (be::sync()) return -1; return ms->barrier.wait() ? 0 : -1; };
    }
    *out = p;
    return 0;
}

static int multi_destroy(demcmc_handle *p)
{
    for (demcmc_handle *k : p->kids) demcmc_destroy(k);
    delete p->multi;
    delete p;
    return 0;
}

// [rows][P_total][w] (host) <- per-kid [rows][P_local][w]
template <class T, class F>
static int multi_interleave(demcmc_handle *p, T *out, int64_t rows, size_t w, F get)
{
    if (!out) return 0;
    const size_t Pt = p->P;
    size_t off = 0;
    for (demcmc_handle *k : p->kids) {
        const size_t Pl = k->P;
        std::vector<T> tmp((size_t)rows * Pl * w);
        if (int rc = get(k, tmp.data())) return rc;
        for (int64_t r = 0; r < rows; ++r) memcpy(out + ((size_t)r * Pt + off) * w, tmp.data() + (size_t)r * Pl * w, sizeof(T) * Pl * w);
        off += Pl;
    }
    return 0;
}

static int multi_history_out(demcmc_handle *p, double *samples, double *lp, uint8_t *accept, int64_t n_rows)
{
    demcmc_handle *k0 = p->kids[0];
    if (n_rows != stored_rows(k0)) return fail(DEMCMC_EINVAL, "n_rows %lld != the %lld stored rows (iterations run / store_every + n_initial)", (long long)n_rows, (long long)stored_rows(k0));
    // one output on the first device, written by every device through peer access, downloaded once
    BE(be::set_device(k0->cfg.device));
    const size_t Pt = p->P, d = p->d;
    double *ds = nullptr, *dl = nullptr; uint8_t *da = nullptr;
    int rc = 0;
    if (samples) ds = (double *)be::dmalloc_shared(sizeof(double) * std::max<size_t>(1, n_rows * Pt * d));
    if (lp) dl = (double *)be::dmalloc_shared(sizeof(double) * std::max<size_t>(1, n_rows * Pt));
    if (accept) da = (uint8_t *)be::dmalloc_shared(std::max<size_t>(1, n_rows * Pt));
    const bool lp_written = p->cfg.update == DEMCMC_UPDATE_MH;
    if ((samples && !ds) || (lp && !dl) || (accept && !da)) rc = fail(DEMCMC_ENOMEM, "output staging does not fit on device %d", k0->cfg.device);
    if (!rc && n_rows > 0) {
        if ((ds && be::dzero(ds, sizeof(double) * n_rows * Pt * d)) || (dl && be::dzero(dl, sizeof(double) * n_rows * Pt)) || (da && be::dzero(da, n_rows * Pt)) || be::sync()) rc = DEMCMC_ECUDA;
        for (demcmc_handle *k : p->kids) {
            if (rc) break;
            if (be::set_device(k->cfg.device) ||
                (stored_rows(k) > 0 && (k->n0 == 0 || k->has_history) &&
                 be::launch_history_by_id(k->hist_theta, k->hist_w, k->hist_acc, k->hist_id, stored_rows(k), 0, n_rows, (int32_t)k->P, (int32_t)d, 0, ds, lp_written ? dl : nullptr, da, (int32_t)Pt)) ||
                be::sync()) rc = DEMCMC_ECUDA;
        }
        if (!rc && be::set_device(k0->cfg.device)) rc = DEMCMC_ECUDA;
        if (!rc && ds && be::d2h(samples, ds, sizeof(double) * n_rows * Pt * d)) rc = DEMCMC_ECUDA;
        if (!rc && dl && be::d2h(lp, dl, sizeof(double) * n_rows * Pt)) rc = DEMCMC_ECUDA;
        if (!rc && da && be::d2h(accept, da, n_rows * Pt)) rc = DEMCMC_ECUDA;
        if (rc == DEMCMC_ECUDA) fail(rc, "history gather: %s", be::last_error());
    }
    be::set_device(k0->cfg.device);
    be::dfree_shared(ds); be::dfree_shared(dl); be::dfree_shared(da);
    return rc;
}

static int multi_get_chains(demcmc_handle *p, int64_t row0, int64_t n_rows, double *out)
{
    demcmc_handle *k0 = p->kids[0];
    if (row0 < 0 || n_rows < 0 || row0 + n_rows > stored_rows(k0)) return fail(DEMCMC_EINVAL, "row range [%lld, %lld) outside the %lld stored rows", (long long)row0, (long long)(row0 + n_rows), (long long)stored_rows(k0));
    if (!k0->has_state) return fail(DEMCMC_ESTATE, "no state");
    if (n_rows == 0) return 0;
    BE(be::set_device(k0->cfg.device));
    const size_t Pt = p->P, d = p->d, n = (size_t)n_rows * Pt * (d + 2);
    double *dout = (double *)be::dmalloc_shared(sizeof(double) * n);
    int32_t *pos = (int32_t *)be::dmalloc_shared(sizeof(int32_t) * Pt);
    int rc = 0;
    if (!dout || !pos) rc = fail(DEMCMC_ENOMEM, "chain staging (%zu MB) does not fit on device %d: %s", sizeof(double) * n >> 20, k0->cfg.device, be::last_error());
    if (!rc && (be::dzero(dout, sizeof(double) * n) || be::sync())) rc = DEMCMC_ECUDA;
    for (int phase = 1; phase <= 2 && !rc; ++phase)           // every device's final positions first, then the rows
        for (demcmc_handle *k : p->kids) {
            if (be::set_device(k->cfg.device) ||
                be::launch_chains(k->hist_theta, k->hist_w, k->hist_acc, k->hist_id, cur_row(k).id, pos, row0, n_rows, (int32_t)k->P, (int32_t)d, 0, dout,
                                  (int32_t)Pt, k->cfg.group_begin * k->cfg.Np, phase) ||
                be::sync()) { rc = DEMCMC_ECUDA; break; }
        }
    if (!rc && (be::set_device(k0->cfg.device) || be::d2h(out, dout, sizeof(double) * n))) rc = DEMCMC_ECUDA;
    if (rc == DEMCMC_ECUDA) fail(rc, "chain gather: %s", be::last_error());
    be::set_device(k0->cfg.device);
    be::dfree_shared(dout); be::dfree_shared(pos);
    return rc;
}

static int multi_get_moments(demcmc_handle *p, int64_t row0, int64_t n_rows, int64_t *count, double *mean, double *m2)
{
    const size_t d = p->d;
    std::vector<double> mk(d), sk(d);
    double ca = 0.0;
    for (size_t k = 0; k < d; ++k) { mean[k] = 0.0; m2[k] = 0.0; }
    for (demcmc_handle *kid : p->kids) {                     // Chan's merge in device order (deterministic)
        int64_t c = 0;
        if (int rc = demcmc_get_moments(kid, row0, n_rows, &c, mk.data(), sk.data())) return rc;
        const double cb = (double)c, cn = ca + cb;
        if (cb > 0)
            for (size_t k = 0; k < d; ++k) {
                const double dl = mk[k] - mean[k];
                mean[k] += dl * (cb / cn);
                m2[k] += sk[k] + dl * dl * (ca * cb / cn);
            }
        ca = cn;
    }
    *count = (int64_t)ca;
    return 0;
}

extern "C" {

const char *demcmc_last_error(void) { return g_err.c_str(); }
int demcmc_abi_version(void) { return DEMCMC_ABI_VERSION; }
int demcmc_device_count(void) { return be::device_count(); }
const char *demcmc_backend_name(void) { return be::name(); }

int demcmc_create(const demcmc_config *cfg, demcmc_handle **out)
{
    if (!cfg || !out) return fail(DEMCMC_EINVAL, "null argument");
    *out = nullptr;
    if (cfg->abi_version != DEMCMC_ABI_VERSION) return fail(DEMCMC_EINVAL, "abi_version %d != %d", cfg->abi_version, DEMCMC_ABI_VERSION);
    if (cfg->n_devices < 0) return fail(DEMCMC_EINVAL, "negative n_devices");
    if (cfg->Np < 3) return fail(DEMCMC_EINVAL, "Np must be >= 3 (two donors besides the target, crossover.jl:158-160)");
    if (cfg->n_groups < 1 || cfg->d < 1 || !cfg->lo || !cfg->hi) return fail(DEMCMC_EINVAL, "bad n_groups/d/bounds");
    if (cfg->n_groups > MAX_MIG) return fail(DEMCMC_EUNSUPPORTED, "n_groups > %d", MAX_MIG);
    if (cfg->n_blocks < 0 || (cfg->n_blocks > 0 && !cfg->blocks)) return fail(DEMCMC_EINVAL, "blocks missing");
    if (cfg->proposal < 0 || cfg->proposal > 2) return fail(DEMCMC_EINVAL, "unknown generate_proposal %d", cfg->proposal);
    if (cfg->store_every < 0) return fail(DEMCMC_EINVAL, "store_every must be >= 1 (0 is read as 1)");
    if (cfg->n_initial < 0 || cfg->donors < 0 || cfg->donors > 1) return fail(DEMCMC_EINVAL, "bad n_initial / donors");
    if (cfg->update < 0 || cfg->update > DEMCMC_UPDATE_MINIMIZE || cfg->fitness < 0 || cfg->fitness > DEMCMC_FITNESS_FUN) return fail(DEMCMC_EINVAL, "unknown update_particle! / evaluate_fitness! kind");
    if (cfg->update != DEMCMC_UPDATE_MH && cfg->theta_snooker != 0.0)
        return fail(DEMCMC_EINVAL, "maximize! / minimize! take no log_adj: with theta_snooker > 0 the reference throws a MethodError (crossover.jl:38)");
    if (cfg->donors == DEMCMC_DONORS_HISTORY) {
        // resample (crossover.jl:113-124) draws from rows 1:de.iter-1: there must be rows to draw from
        if ((int64_t)cfg->n_initial * cfg->n_groups * cfg->Np < 3) return fail(DEMCMC_EINVAL, "sample = resample needs n_initial prior rows (at least 3 stored particles)");
    }
    if (cfg->n_devices > 1) return multi_create(cfg, out);
    if (be::device_count() <= 0) return fail(DEMCMC_ENODEVICE, "no CUDA device: libdemcmc_b200 has no CPU fallback (%s)", be::last_error());
    const int dev0 = (cfg->n_devices == 1 && cfg->devices) ? cfg->devices[0] : cfg->device;
    if (be::set_device(dev0) != 0) return fail(DEMCMC_ENODEVICE, "cannot select device %d: %s", cfg->device, be::last_error());

    demcmc_handle *h = new demcmc_handle();
    h->cfg = *cfg;
    h->cfg.device = dev0; h->cfg.n_devices = 0; h->cfg.devices = nullptr;
    h->d = cfg->d;
    h->n0 = cfg->n_initial;
    h->k_store = std::max(1, cfg->store_every);
    h->n_scratch = (h->k_store > 1 || cfg->n_blocks > 0) ? MAX_CHUNK + 2 : 3;      // chunks of overlapped block sweeps write scratch rows too
    // long parameter vectors (the wide kernels, one CTA per particle): two chains of kernels over two halves of the groups
    // overlap one half's latency-bound likelihood launch with the other's issue-bound proposals (configs[3]: 21.7 -> 23.7 M
    // updates/s; 3 / 4 lanes: 19.3 / 18.4; configs[4]'s shard, d = 101: no gain)
    if (cfg->d >= 256) h->n_lanes = 2;
    if (const char *e = getenv("DEMCMC_LANES")) h->n_lanes = std::max(1, std::min<int>(atoi(e), be::MAX_LANES));   // A/B measurements
    h->G_local = cfg->group_count > 0 ? cfg->group_count : cfg->n_groups;
    if (cfg->group_begin < 0 || cfg->group_begin + h->G_local > cfg->n_groups) { delete h; return fail(DEMCMC_EINVAL, "group shard out of range"); }
    h->P = h->G_local * cfg->Np;
    h->B = cfg->n_blocks > 0 ? cfg->n_blocks : 1;
    h->lo.assign(cfg->lo, cfg->lo + cfg->d);
    h->hi.assign(cfg->hi, cfg->hi + cfg->d);
    if (cfg->n_blocks > 0) h->blocks.assign(cfg->blocks, cfg->blocks + (size_t)cfg->n_blocks * cfg->d);
    if (cfg->n_groups == 1) h->cfg.alpha = 0.0;   // structs.jl:102-105
    memset(&h->ctr, 0, sizeof h->ctr);
    memset(&h->dmodel, 0, sizeof h->dmodel);
    h->group_owner.assign(cfg->n_groups, 0);

    const size_t P = h->P, d = h->d;
    h->d_lo = (double *)be::dmalloc(sizeof(double) * d);
    h->d_hi = (double *)be::dmalloc(sizeof(double) * d);
    h->d_blocks = (uint8_t *)be::dmalloc(std::max<size_t>(1, h->blocks.size()));
    h->scr_theta = (double *)be::dmalloc(sizeof(double) * h->n_scratch * P * d);
    h->scr_w = (double *)be::dmalloc(sizeof(double) * h->n_scratch * P);
    h->scr_id = (int32_t *)be::dmalloc(sizeof(int32_t) * h->n_scratch * P);
    h->scr_acc = (uint8_t *)be::dmalloc((size_t)h->n_scratch * P);
    h->prop_theta = (double *)be::dmalloc(sizeof(double) * P * d);
    h->prop_prior = (double *)be::dmalloc(sizeof(double) * P);
    h->prop_adj = (double *)be::dmalloc(sizeof(double) * P);
    h->prop_msq = (double *)be::dmalloc(sizeof(double) * P);
    h->prop_inb = (uint8_t *)be::dmalloc(P);
    {
        // only where one CTA per particle repeats the draws in every warp (the wide kernels, d >= 256: +1 % on configs[3]);
        // with one warp per particle the launch costs more than it saves (configs[0]: -6 %).  DEMCMC_PLAN=1 / 0 forces it.
        const char *e = getenv("DEMCMC_PLAN");
        const bool on = e ? e[0] == '1' : d >= 256;
        if (on) h->plan_recs = (PlanRec *)be::dmalloc(sizeof(PlanRec) * (size_t)MAX_CHUNK * P);
    }
    h->ll_acc = (long long *)be::dmalloc(sizeof(long long) * P);
    h->ll_q = (double *)be::dmalloc(sizeof(double) * P);
    h->base_th = (double *)be::dmalloc(sizeof(double) * P);
    h->base_cw = (double *)be::dmalloc(sizeof(double) * P);
    h->base_tot = (double *)be::dmalloc(sizeof(double) * std::max(1, h->G_local));
    h->d_picks = (int32_t *)be::dmalloc(sizeof(int32_t) * MAX_MIG);
    h->d_stage = (double *)be::dmalloc(sizeof(double) * MAX_MIG * (d + 3));
    h->d_stage_recv = (double *)be::dmalloc(sizeof(double) * MAX_MIG * (d + 3));
    bool ok = h->d_lo && h->d_hi && h->d_blocks && h->scr_theta && h->scr_w && h->scr_id && h->scr_acc && h->prop_theta &&
              h->prop_prior && h->prop_adj && h->prop_msq && h->prop_inb && h->ll_acc && h->ll_q && h->base_th && h->base_cw && h->base_tot && h->d_picks && h->d_stage && h->d_stage_recv;
    for (int i = 0; i < demcmc_handle::RING && ok; ++i) {
        Upload &u = h->ring[i];
        u.off_mut = sizeof(SweepCtx) * MAX_CHUNK;
        u.off_order = (u.off_mut + (size_t)h->G_local * MAX_CHUNK + 63) & ~(size_t)63;
        u.bytes = u.off_order + sizeof(int32_t) * P * MAX_CHUNK;
        u.h_blk = (uint8_t *)be::hmalloc_pinned(u.bytes);
        u.d_blk = (uint8_t *)be::dmalloc(u.bytes);
        u.copied = be::event_create();
        ok = u.h_blk && u.d_blk && u.copied;
        if (ok) {
            u.h_ctx = (SweepCtx *)u.h_blk; u.h_mut = u.h_blk + u.off_mut; u.h_order = (int32_t *)(u.h_blk + u.off_order);
            u.d_ctx = (SweepCtx *)u.d_blk; u.d_mut = u.d_blk + u.off_mut; u.d_order = (int32_t *)(u.d_blk + u.off_order);
        }
    }
    if (!ok) { demcmc_destroy(h); return fail(DEMCMC_ENOMEM, "device allocation failed: %s", be::last_error()); }
    if (be::h2d(h->d_lo, h->lo.data(), sizeof(double) * d) || be::h2d(h->d_hi, h->hi.data(), sizeof(double) * d) ||
        (!h->blocks.empty() && be::h2d(h->d_blocks, h->blocks.data(), h->blocks.size())) || be::sync()) {
        demcmc_destroy(h);
        return fail(DEMCMC_ECUDA, "upload failed: %s", be::last_error());
    }
    ConfigDev &c = h->dcfg;
    c.Np = cfg->Np; c.d = cfg->d; c.G_local = h->G_local; c.group_begin = cfg->group_begin; c.proposal = cfg->proposal;
    c.burnin = cfg->burnin; c.n_blocks = cfg->n_blocks; c.eps = cfg->eps; c.sigma = cfg->sigma; c.kappa = cfg->kappa;
    c.resample = cfg->donors; c.P_hist = h->P; c.update = cfg->update; c.fitness = cfg->fitness; c.theta_snooker = cfg->theta_snooker; c.lo = h->d_lo; c.hi = h->d_hi; c.blocks = h->d_blocks; c.seed = cfg->seed;
    *out = h;
    return 0;
}

int demcmc_destroy(demcmc_handle *h)
{
    if (!h) return 0;
    if (h->multi) return multi_destroy(h);
    be::set_device(h->cfg.device);
    be::sync();
    if (!h->mbox_shared) { for (Mbox &m : h->peer_maps) be::mbox_close(&m); be::mbox_destroy(&h->mbox); }
    be::timeline_dump();
    be::dfree(h->ghist_theta); be::dfree(h->ghist_pos); be::dfree(h->gid_tmp);
    if (h->comm) be::comm_destroy(h->comm);
    for (void *p : h->model_allocs) be::dfree(p);
    if (h->custom_mod) be::custom_unload(h->custom_mod);
    void *ptrs[] = { h->hist_theta, h->hist_w, h->hist_id, h->hist_acc, h->hist_pos, h->scr_theta, h->scr_w, h->scr_id, h->scr_acc,
                     h->prop_theta, h->prop_prior, h->prop_adj, h->prop_msq, h->prop_inb, h->ll_acc, h->ll_q, h->base_th, h->base_cw, h->base_tot, h->ll_part, h->d_lo, h->d_hi, h->d_blocks,
                     h->plan_recs, h->d_picks, h->d_stage, h->d_stage_recv, h->d_mig_log, h->tr_theta, h->tr_w, h->tr_adj, h->tr_xdot, h->tr_acc, h->flush_buf };
    for (void *e : h->tev) be::tevent_destroy(e);
    for (void *p : ptrs) be::dfree(p);
    for (auto &u : h->ring) { be::hfree_pinned(u.h_blk); be::dfree(u.d_blk); be::event_destroy(u.copied); }
    delete h;
    return 0;
}

static_assert(CUSTOM_MAX_PAR == DEMCMC_CUSTOM_MAX_PAR, "k_ll_custom stages DEMCMC_CUSTOM_MAX_PAR values per particle");
static const char NO_CUSTOM[] = "custom likelihoods need the CUDA backend (this backend has no run-time compiler)";

int demcmc_set_model(demcmc_handle *h, const demcmc_model *m)
{
    if (!h || !m || !m->prior) return fail(DEMCMC_EINVAL, "null argument");
    if (h->multi) {
        const int rc = for_kids(h, [&](demcmc_handle *k, int) { return demcmc_set_model(k, m); });
        if (!rc) { h->has_model = true; h->dmodel = h->kids[0]->dmodel; }
        return rc;
    }
    if (m->d != h->d) return fail(DEMCMC_EINVAL, "model.d %d != config.d %d", m->d, h->d);
    BE(be::set_device(h->cfg.device));
    for (void *p : h->model_allocs) be::dfree(p);
    h->model_allocs.clear();
    if (h->custom_mod) {                                     // rebinding: no launch may still use the old module
        BE(be::sync());
        be::custom_unload(h->custom_mod);
        h->custom_mod = nullptr;
    }
    be::dfree(h->ll_part); h->ll_part = nullptr;
    ModelDev &D = h->dmodel;
    memset(&D, 0, sizeof D);
    D.kind = m->kind; D.d = m->d; D.n_obs = m->n_obs; D.n_dim = m->n_dim; D.n_per = m->n_per; D.lba_floor = m->lba_floor;
    auto upload = [&](const void *src, size_t bytes, bool on_dev) -> void * {
        void *p = be::dmalloc(std::max<size_t>(bytes, 8));
        if (!p) return nullptr;
        h->model_allocs.push_back(p);
        if (bytes && (on_dev ? be::d2d(p, src, bytes) : be::h2d(p, src, bytes))) return nullptr;
        return p;
    };
    // parameter-count contract of each registered kernel
    int want_d = -1;
    switch (m->kind) {
    case DEMCMC_GAUSSIAN: want_d = 2; break;
    case DEMCMC_MVNORMAL: want_d = m->n_dim + 1; break;
    case DEMCMC_BINOMIAL: want_d = 1; break;
    case DEMCMC_LNR: want_d = m->n_dim + 1; break;
    case DEMCMC_LBA: want_d = m->n_dim + 3; break;
    case DEMCMC_HIER_NORMAL: want_d = m->n_dim + 3; break;
    case DEMCMC_RASTRIGIN: want_d = m->d; break;
    case DEMCMC_MVNORMAL_FULL: want_d = m->n_dim + 1; break;
    case DEMCMC_CUSTOM:
        if (!be::custom_load) return fail(DEMCMC_EUNSUPPORTED, "%s", NO_CUSTOM);
        if (m->d < 1 || m->d > DEMCMC_CUSTOM_MAX_PAR) return fail(DEMCMC_EUNSUPPORTED, "a custom likelihood takes 1..%d parameters, got d = %d", DEMCMC_CUSTOM_MAX_PAR, m->d);
        if (!m->source) return fail(DEMCMC_EINVAL, "a custom likelihood needs model.source");
        if (m->n_obs > 0 && m->n_cols < 1) return fail(DEMCMC_EINVAL, "a custom likelihood with observations needs n_cols >= 1, got %d", m->n_cols);
        want_d = m->d;
        break;
    default: return fail(DEMCMC_EUNSUPPORTED, "no registered kernel for model kind %d: arbitrary closures are not supported and there is no CPU fallback", m->kind);
    }
    if (m->d != want_d) return fail(DEMCMC_EINVAL, "model kind %d expects d = %d, got %d", m->kind, want_d, m->d);
    if (!m->x && m->kind != DEMCMC_RASTRIGIN && !(m->kind == DEMCMC_CUSTOM && m->n_obs == 0)) return fail(DEMCMC_EINVAL, "model data missing");
    if ((m->kind == DEMCMC_LNR || m->kind == DEMCMC_LBA) && (!m->choice || m->n_dim < 2 || m->n_dim > MAX_ACC))
        return fail(DEMCMC_EINVAL, "LNR/LBA need choices and 2..%d accumulators", MAX_ACC);
    if (m->n_obs < 0) return fail(DEMCMC_EINVAL, "negative n_obs");

    std::vector<Prior> pr(m->d);
    for (int k = 0; k < m->d; ++k) {
        pr[k].kind = m->prior[k].kind; pr[k].ref = m->prior[k].ref; pr[k].a = m->prior[k].a; pr[k].b = m->prior[k].b;
        if (pr[k].kind < 0 || pr[k].kind > PRIOR_NORMAL_REF) return fail(DEMCMC_EUNSUPPORTED, "prior kind %d of parameter %d is not registered", pr[k].kind, k);
        if (pr[k].kind == PRIOR_NORMAL_REF && (pr[k].ref < 0 || pr[k].ref >= m->d)) return fail(DEMCMC_EINVAL, "prior ref out of range");
        if (pr[k].kind == PRIOR_NORMAL_REF) D.prior_has_ref = 1;
        prior_constants(pr[k]);
    }
    D.prior = (const Prior *)upload(pr.data(), sizeof(Prior) * pr.size(), false);
    if (!D.prior) return fail(DEMCMC_ENOMEM, "prior upload failed");
    const bool dev = m->data_on_device != 0;
    D.n_osplit = 1; D.n_ksplit = 1; D.split_len = 0; D.ksplit_len = 0;
    if (m->kind == DEMCMC_RASTRIGIN) {
        D.n_obs = 0;                                  // an objective of the parameters alone (optimize path)
    } else if (m->kind == DEMCMC_BINOMIAL) {
        double nk[2];
        if (dev) { BE(be::d2h(nk, m->x, sizeof nk)); } else memcpy(nk, m->x, sizeof nk);
        D.binom_N = nk[0]; D.binom_k = nk[1]; D.n_obs = 1;
    } else if (m->kind == DEMCMC_MVNORMAL || m->kind == DEMCMC_HIER_NORMAL || m->kind == DEMCMC_MVNORMAL_FULL) {
        // SSD layout: xT[k][ld]; MVN: k = dimension, obs = n_obs; hierarchical: k = subject, obs = n_per
        D.ssd_k = m->n_dim;
        D.ssd_n = m->kind == DEMCMC_HIER_NORMAL ? m->n_per : m->n_obs;
        if (m->kind == DEMCMC_HIER_NORMAL) D.n_obs = (int64_t)m->n_dim * m->n_per;
        D.ssd_ld = (D.ssd_n + SSD_TN - 1) / SSD_TN * SSD_TN;
        if (D.ssd_ld == 0) D.ssd_ld = SSD_TN;
        // dimension splits: balanced, at most SSD_KS dimensions (SSD_NJ DMMA k-steps) each
        D.n_ksplit = (D.ssd_k + SSD_KS - 1) / SSD_KS;
        D.ksplit_len = (D.ssd_k + D.n_ksplit - 1) / D.n_ksplit;
        D.ssd_nj = (D.ksplit_len + 3) / 4;
        D.ksplit_magic = (uint32_t)((((uint64_t)1 << 32) + (uint64_t)D.ksplit_len - 1) / (uint64_t)D.ksplit_len);
        { const char *e = getenv("DEMCMC_NO_HALF_STEP"); D.ssd_half = (D.ksplit_len % 4 == 2 && !(e && e[0] == '1')) ? 1 : 0; }
        { const char *e = getenv("DEMCMC_TEST_CORRUPT"); D.debug_corrupt = e ? atoi(e) : 0; }     // mutation tests (de_types.h)
        D.center_given = m->center ? 1 : 0;
        if (h->suffstat && m->center) return fail(DEMCMC_EINVAL, "sufficient-statistic mode needs the data centred on their column means (model.center = NULL)");
        D.n_osplit = 1; D.split_len = (int32_t)std::min<int64_t>(D.ssd_ld, INT32_MAX);
        // fixed-point bits below the per-particle bound: the sum of one rounded term per
        // (observation row, dimension split) must stay below 2^62
        int64_t terms = D.ssd_ld * D.n_ksplit;
        int lg = 0;
        while (((int64_t)1 << lg) < terms) ++lg;
        D.ssd_qbits = std::min(50, 62 - lg);
        double *xT = (double *)be::dmalloc(sizeof(double) * std::max(be::pack_ssd_doubles(D), (size_t)D.ssd_k * D.ssd_ld));
        double *center = (double *)be::dmalloc(sizeof(double) * (size_t)D.ssd_k);
        if (!xT || !center) return fail(DEMCMC_ENOMEM, "data do not fit on the device");
        h->model_allocs.push_back(xT);
        h->model_allocs.push_back(center);
        D.xT = xT;
        D.center = center;
        if (m->kind == DEMCMC_MVNORMAL_FULL) {
            // MvNormal(mu, sigma^2 Sigma), Sigma known: Cholesky Sigma = L L', the data whitened once (y = L^-1 x), and the
            // device keeps L^-1 to whiten every proposal's mean when it is staged (de_particle.h: centred_mean)
            const int k = m->n_dim;
            if (!m->cov) return fail(DEMCMC_EINVAL, "MVNORMAL_FULL needs model.cov");
            if (dev) return fail(DEMCMC_EUNSUPPORTED, "MVNORMAL_FULL whitens the data on the host: pass host data");
            if (k < 1 || k > 1024) return fail(DEMCMC_EUNSUPPORTED, "MVNORMAL_FULL supports 1..1024 dimensions");
            std::vector<double> L((size_t)k * k, 0.0), Li((size_t)k * k, 0.0);
            double logdet = 0.0;
            for (int i = 0; i < k; ++i)
                for (int j = 0; j <= i; ++j) {
                    if (fabs(m->cov[(size_t)i * k + j] - m->cov[(size_t)j * k + i]) > 1e-12 * (fabs(m->cov[(size_t)i * k + i]) + fabs(m->cov[(size_t)j * k + j])))
                        return fail(DEMCMC_EINVAL, "model.cov is not symmetric at (%d, %d)", i, j);
                    long double sacc = m->cov[(size_t)i * k + j];
                    for (int q = 0; q < j; ++q) sacc -= (long double)L[(size_t)i * k + q] * L[(size_t)j * k + q];
                    if (i == j) {
                        if (!(sacc > 0)) return fail(DEMCMC_EINVAL, "model.cov is not positive definite (pivot %d)", i);
                        L[(size_t)i * k + i] = sqrt((double)sacc);
                        logdet += 2.0 * log(L[(size_t)i * k + i]);
                    } else L[(size_t)i * k + j] = (double)(sacc / L[(size_t)j * k + j]);
                }
            for (int c = 0; c < k; ++c)                          // L^-1 column by column: L z = e_c
                for (int r = c; r < k; ++r) {
                    long double t = r == c ? 1.0L : 0.0L;
                    for (int q = c; q < r; ++q) t -= (long double)L[(size_t)r * k + q] * Li[(size_t)q * k + c];
                    Li[(size_t)r * k + c] = (double)(t / L[(size_t)r * k + r]);
                }
            std::vector<double> y((size_t)m->n_obs * k);
            for (int64_t i = 0; i < m->n_obs; ++i) {
                const double *xi = m->x + (size_t)i * k;
                double *yi = y.data() + (size_t)i * k;
                for (int r = 0; r < k; ++r) {                    // forward substitution: the same arithmetic as whitening through L
                    long double t = xi[r];
                    for (int q = 0; q < r; ++q) t -= (long double)L[(size_t)r * k + q] * yi[q];
                    yi[r] = (double)(t / L[(size_t)r * k + r]);
                }
            }
            D.linv = (const double *)upload(Li.data(), sizeof(double) * Li.size(), false);
            if (!D.linv) return fail(DEMCMC_ENOMEM, "covariance factor upload failed");
            D.logdet = logdet;
            BE(be::launch_pack_ssd(y.data(), 0, m->center, &D));
        } else
        BE(be::launch_pack_ssd(m->x, dev, m->center, &D));       // centres and packs the data, fills D.ssd_xx / D.ssd_rowmax
    } else {
        // the pointwise kinds, and DEMCMC_CUSTOM: x[n_obs][n_cols], through the same observation splits (k_ll_custom).
        // A custom model never qualifies for the fused / small-chunk / persistent kernels (their densities are the
        // registered ones): every level runs propose -> k_ll_custom -> accept
        const int64_t n_val = m->n_obs * (m->kind == DEMCMC_CUSTOM ? (int64_t)m->n_cols : 1);
        D.x = (const double *)upload(m->x, sizeof(double) * n_val, dev);
        if (!D.x) return fail(DEMCMC_ENOMEM, "data upload failed");
        if (m->kind == DEMCMC_CUSTOM) {
            D.n_cols = m->n_cols;
            int has_obs = 0;
            if (int rc = be::custom_load(m->source, &h->custom_mod, &has_obs)) {
                g_err = be::last_error();                    // the whole compiler log (fail() would cut it)
                return rc == -1 ? DEMCMC_EINVAL : rc == -2 ? DEMCMC_EUNSUPPORTED : DEMCMC_ECUDA;
            }
            if (m->n_obs > 0 && !has_obs)
                return fail(DEMCMC_EINVAL, "the model has %lld observations but its source defines no "
                            "__device__ double demcmc_obs(const double *par, const double *x)", (long long)m->n_obs);
            D.custom = h->custom_mod;
        }
        if (m->choice) { D.choice = (const int32_t *)upload(m->choice, sizeof(int32_t) * m->n_obs, dev); if (!D.choice) return fail(DEMCMC_ENOMEM, "data upload failed"); }
        if (m->sigma) { D.has_sigma = 1; for (int r = 0; r < m->n_dim && r < MAX_ACC; ++r) D.sigma_acc[r] = m->sigma[r]; }
        const int64_t chunk = PW_THREADS;
        const int64_t chunks = std::max<int64_t>(1, (m->n_obs + chunk - 1) / chunk);
        const int64_t per = std::max<int64_t>(1, (chunks + 147) / 148);
        D.split_len = (int32_t)(per * chunk);
        D.n_osplit = (int32_t)std::max<int64_t>(1, (m->n_obs + D.split_len - 1) / D.split_len);
    }
    const size_t n_split = (size_t)D.n_osplit * D.n_ksplit;
    h->ll_part = (double *)be::dmalloc(sizeof(double) * std::max<size_t>(1, (size_t)h->P * n_split));
    if (!h->ll_part) return fail(DEMCMC_ENOMEM, "partial-sum workspace does not fit");
    BE(be::sync());
    h->has_model = true;
    return 0;
}

int demcmc_compile_loglike(const char *source, char *log, int64_t log_cap)
{
    if (log && log_cap > 0) log[0] = 0;
    if (!source) return fail(DEMCMC_EINVAL, "null source");
    if (!be::custom_compile) return fail(DEMCMC_EUNSUPPORTED, "%s", NO_CUSTOM);
    const int rc = be::custom_compile(source);
    if (rc == 0) return 0;
    g_err = be::last_error();                                // the whole compiler log (fail() would cut it)
    if (log && log_cap > 0) { const size_t n = std::min(g_err.size(), (size_t)log_cap - 1); memcpy(log, g_err.data(), n); log[n] = 0; }
    return rc == -2 ? DEMCMC_EUNSUPPORTED : DEMCMC_EINVAL;
}

int demcmc_set_history(demcmc_handle *h, const double *rows)
{
    if (!h || !rows) return fail(DEMCMC_EINVAL, "null argument");
    if (h->n0 <= 0) return fail(DEMCMC_EINVAL, "the handle was created with n_initial = 0");
    if (h->iters_done > 0) return fail(DEMCMC_ESTATE, "set_history must come before the first run");
    if (h->multi) {                                          // rows[n_initial][P_total][d] -> every device its own ids
        const size_t Pt = h->P, dd = h->d;
        const int rc = for_kids(h, [&](demcmc_handle *k, int) {
            if (h->cfg.donors) return demcmc_set_history(k, rows);    // sample = resample: every device keeps the rows of ALL ids
            const size_t Pl = k->P, pb = (size_t)k->cfg.group_begin * k->cfg.Np;
            std::vector<double> part((size_t)h->n0 * Pl * dd);
            for (int64_t r = 0; r < h->n0; ++r) memcpy(part.data() + (size_t)r * Pl * dd, rows + ((size_t)r * Pt + pb) * dd, sizeof(double) * Pl * dd);
            return demcmc_set_history(k, part.data());
        });
        if (!rc) h->has_history = true;
        return rc;
    }
    // sample = resample on a sharded job: rows of ALL ids (the donors' history is replicated); otherwise the
    // rows of the handle's own particles
    const bool sharded = h->G_local != h->cfg.n_groups && h->cfg.donors;
    if (sharded && h->n_ranks <= 1) return fail(DEMCMC_ESTATE, "initial history rows of a sharded resample job: demcmc_comm_init must come first");
    BE(be::set_device(h->cfg.device));
    if (int rc = grow_history(h, h->n0)) return rc;
    const size_t P = h->P, d = h->d, n = (size_t)h->n0 * P;
    const size_t Pt = (size_t)h->cfg.n_groups * h->cfg.Np, pbeg = (size_t)h->cfg.group_begin * h->cfg.Np;
    // initialize_samples (utilities.jl:35-39): samples[i, :, p] by particle id; before any
    // migration id == position, accept = false and lp = 0.0 (utilities.jl:18-20).  A sharded job
    // passes the rows of ALL ids ([n_initial][P_total][d]): its slice is this rank's history, the
    // whole is the replicated copy the donors are drawn from.
    std::vector<int32_t> idv(n);
    for (size_t i = 0; i < n; ++i) idv[i] = (int32_t)(pbeg + i % P);
    if (!sharded) BE(be::h2d(h->hist_theta, rows, sizeof(double) * n * d));
    else {
        for (int64_t r = 0; r < h->n0; ++r) BE(be::h2d(h->hist_theta + (size_t)r * P * d, rows + ((size_t)r * Pt + pbeg) * d, sizeof(double) * P * d));
        std::vector<int32_t> gid((size_t)h->n0 * Pt);
        for (size_t i = 0; i < gid.size(); ++i) gid[i] = (int32_t)(i % Pt);
        BE(be::h2d(h->ghist_theta, rows, sizeof(double) * (size_t)h->n0 * Pt * d));
        BE(be::h2d(h->ghist_pos, gid.data(), sizeof(int32_t) * gid.size()));
    }
    BE(be::h2d(h->hist_id, idv.data(), sizeof(int32_t) * n));
    if (h->hist_pos) { for (size_t i = 0; i < n; ++i) idv[i] = (int32_t)(i % P); BE(be::h2d(h->hist_pos, idv.data(), sizeof(int32_t) * n)); }
    BE(be::dzero(h->hist_w, sizeof(double) * n));
    BE(be::dzero(h->hist_acc, n));
    BE(be::sync());
    h->has_history = true;
    return 0;
}

int demcmc_set_state(demcmc_handle *h, const double *theta, const int32_t *ids)
{
    if (!h) return fail(DEMCMC_EINVAL, "null argument");
    if (!theta && !(h->n0 > 0 && h->has_history)) return fail(DEMCMC_EINVAL, "null theta (allowed only after demcmc_set_history: init_particle then starts from samples[1, :, id])");
    if (!h->has_model) return fail(DEMCMC_ESTATE, "set_model must come before set_state");
    if (h->multi) {
        const int rc = for_kids(h, [&](demcmc_handle *k, int) {
            const size_t pb = (size_t)k->cfg.group_begin * k->cfg.Np;
            return demcmc_set_state(k, theta ? theta + pb * h->d : nullptr, ids ? ids + pb : nullptr);
        });
        if (!rc) h->has_state = true;
        return rc;
    }
    BE(be::set_device(h->cfg.device));
    const size_t P = h->P, d = h->d;
    // the current state moves to scratch row 0 (history rows already written stay as they are)
    h->cur_hist = -1; h->cur_scratch = 0; h->scr_cursor = 0;
    Row r = row_of(h, false, 0);
    std::vector<int32_t> idv(P);
    for (size_t p = 0; p < P; ++p) idv[p] = ids ? ids[p] : (int32_t)(h->cfg.group_begin * h->cfg.Np + p);
    if (theta) BE(be::h2d(r.theta, theta, sizeof(double) * P * d));
    else BE(be::d2d(r.theta, h->hist_theta, sizeof(double) * P * d));       // utilities.jl:15
    BE(be::h2d(r.id, idv.data(), sizeof(int32_t) * P));
    BE(be::dzero(r.acc, P));
    BE(be::sync());
    // init_particle (utilities.jl:13-22): weight through evaluate_fitness!
    BE(be::launch_eval(h->dcfg, h->dmodel, r.theta, (int64_t)P, nullptr, nullptr, r.w, h->ll_part));
    BE(be::sync());
    h->has_state = true;
    return 0;
}

namespace {
// The local shard of a replay tape: the device arrays the sweep contexts point into and the host copies the planner
// reads.  It owns its device buffers, so every return out of a run frees them.
struct TapeShard {
    uint8_t *t_kind = nullptr, *t_keep = nullptr;
    int32_t *t_idx = nullptr, *t_idx_row = nullptr;
    double *t_g1 = nullptr, *t_g2 = nullptr, *t_uacc = nullptr, *t_noise = nullptr;
    std::vector<uint8_t> hk; std::vector<int32_t> hi;             // host copies of the local kinds and idx, for the planner
    TapeShard() = default; TapeShard(const TapeShard &) = delete; TapeShard &operator=(const TapeShard &) = delete;
    ~TapeShard() { for (void *p : { (void *)t_kind, (void *)t_idx, (void *)t_idx_row, (void *)t_g1, (void *)t_g2, (void *)t_uacc, (void *)t_noise, (void *)t_keep }) be::dfree(p); }
};

// what the steps of one run_impl call share
struct RunCall {
    const demcmc_tape *tape = nullptr;                            // replay, else nullptr
    TapeShard shard;
    int64_t n_iter = 0, S = 0;
    bool ghist = false;                                           // donors come from the replicated history
    bool skip_stream = false;                                     // the likelihood needs no O(N d) stream (demcmc_set_sufficient_stat)
    int persist_lanes = 0, n_lanes = 1;                           // lanes of the persistent chunk kernel (0: not used), lanes launched
    std::vector<std::pair<int64_t, int>> mig_events;              // iterations that migrated, and how many groups
    // timing events: one pair per chunk when the L2 flush is on; the likelihood launches get their own pairs after those
    size_t tev_ll0 = 0, tev_ll = 0, tev_chunks = 0;
    int64_t n_levels = 0, sweeps_run = 0, chunks_this_call = 0;
    double host_plan_s = 0.0, host_chunk_s = 0.0;
    ChunkPlan plans[be::MAX_LANES];
};

// one chunk: `n_sw` consecutive sweeps starting at local iteration it0 (block b0), staged in ring slot u; lane_off[ln]:
// the first entry of lane ln in u.d_order
struct Chunk { int64_t it0; int b0, n_sw; bool blocked; Upload &u; bool basedep[MAX_CHUNK]; int32_t lane_off[be::MAX_LANES + 1]; };

// DEMCMC_HOST_PROFILE=1: host seconds spent planning and launching, printed per call (stderr)
bool host_profile() { static const bool on = [] { const char *e = getenv("DEMCMC_HOST_PROFILE"); return e && e[0] == '1'; }(); return on; }
double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
struct HostTimer { double &acc; const double t0 = host_profile() ? now_s() : 0.0; ~HostTimer() { if (host_profile()) acc += now_s() - t0; } };
} // namespace

// validates a replay tape and uploads this handle's shard of it
static int load_tape(demcmc_handle *h, const demcmc_tape *tape, int64_t n_iter, TapeShard &ts)
{
    const demcmc_config &cfg = h->cfg;
    const int Np = cfg.Np, Gt = cfg.n_groups, P = h->P, d = h->d, B = h->B;
    const int64_t Pt = (int64_t)Gt * Np, S = n_iter * B, pbeg = (int64_t)cfg.group_begin * Np;
    if (!tape->kind || !tape->idx || !tape->gamma1 || !tape->gamma2 || !tape->u_acc || !tape->noise)
        return fail(DEMCMC_EINVAL, "tape misses a required array");
    if (cfg.kappa != 1.0 && !tape->keep) return fail(DEMCMC_EINVAL, "kappa != 1 needs tape.keep");
    if (Gt > 1 && (!tape->mig_n || !tape->mig_groups || !tape->mig_pick_u)) return fail(DEMCMC_EINVAL, "tape misses the migration arrays");
    if (cfg.donors && !tape->idx_row) return fail(DEMCMC_EINVAL, "sample = resample needs tape.idx_row");
    auto slice = [&](const auto *src, size_t per) {           // [S][Pt][per] -> [S][P][per]
        std::vector<std::remove_const_t<std::remove_reference_t<decltype(*src)>>> v((size_t)S * P * per);
        for (int64_t s = 0; s < S; ++s) std::copy_n(src + ((size_t)s * Pt + pbeg) * per, (size_t)P * per, v.data() + (size_t)s * P * per);
        return v;
    };
    auto upload = [](auto *&dst, const auto &v) {
        const size_t bytes = sizeof v[0] * v.size();
        dst = (std::remove_reference_t<decltype(dst)>)be::dmalloc(std::max<size_t>(8, bytes));
        return dst && (!bytes || !(be::h2d(dst, v.data(), bytes) || be::sync()));
    };
    ts.hk = slice(tape->kind, 1); ts.hi = slice(tape->idx, 3);
    if (!upload(ts.t_kind, ts.hk) || !upload(ts.t_idx, ts.hi) || (cfg.donors && !upload(ts.t_idx_row, slice(tape->idx_row, 3))) ||
        !upload(ts.t_g1, slice(tape->gamma1, 1)) || !upload(ts.t_g2, slice(tape->gamma2, 1)) || !upload(ts.t_uacc, slice(tape->u_acc, 1)) ||
        !upload(ts.t_noise, slice(tape->noise, d)) || (cfg.kappa != 1.0 && !upload(ts.t_keep, slice(tape->keep, d))))
        return fail(DEMCMC_ENOMEM, "tape upload failed: %s", be::last_error());
    const std::vector<uint8_t> &hk = ts.hk; const std::vector<int32_t> &hi = ts.hi;
    for (size_t i = 0; i < hk.size(); ++i) if (hk[i] > KIND_MUTATION) return fail(DEMCMC_EINVAL, "tape.kind[%zu] = %d", i, hk[i]);
    for (size_t i = 0; i < hi.size(); ++i) {
        const uint8_t k = hk[i / 3];
        if (k == KIND_MUTATION) continue;
        const bool base = k == KIND_DE && i % 3 == 0;          // slot of the base particle in the group, or -1
        if (base && hi[i] < 0) continue;
        const int64_t lim = (cfg.donors && !base) ? Pt : Np;   // resample donors are particle ids
        if (hi[i] < 0 || hi[i] >= lim) return fail(DEMCMC_EINVAL, "tape.idx[%zu] = %d out of range", i, hi[i]);
        if (cfg.donors && !base) {
            const int64_t sw = (int64_t)(i / 3) / P, pl = (int64_t)(i / 3) % P;
            const int64_t ub = stored_rows(h, h->iters_done + sw / B);                   // rows 1:de.iter-1
            const int32_t r = tape->idx_row[((size_t)sw * Pt + pbeg + pl) * 3 + i % 3];
            if (r < 0 || r >= ub) return fail(DEMCMC_EINVAL, "tape.idx_row of sweep %lld particle %lld = %d outside the %lld stored rows", (long long)sw, (long long)pl, r, (long long)ub);
        }
    }
    return 0;
}

// the trace and the migration log of this call
static int reset_call_buffers(demcmc_handle *h, const RunCall &call)
{
    const int64_t S = call.S, n_iter = call.n_iter; const size_t P = h->P, d = h->d;
    be::dfree(h->tr_theta); be::dfree(h->tr_w); be::dfree(h->tr_adj); be::dfree(h->tr_acc); be::dfree(h->tr_xdot);
    h->tr_theta = h->tr_w = h->tr_adj = h->tr_xdot = nullptr; h->tr_acc = nullptr; h->tr_sweeps = 0;
    const bool ssd_model = is_ssd(h->dmodel.kind);
    if (h->cfg.trace && S > 0) {
        h->tr_theta = (double *)be::dmalloc(sizeof(double) * S * P * d);
        h->tr_w = (double *)be::dmalloc(sizeof(double) * S * P);
        h->tr_adj = (double *)be::dmalloc(sizeof(double) * S * P);
        h->tr_acc = (uint8_t *)be::dmalloc((size_t)S * P);
        if (ssd_model) h->tr_xdot = (double *)be::dmalloc(sizeof(double) * S * P);
        if (!h->tr_theta || !h->tr_w || !h->tr_adj || !h->tr_acc || (ssd_model && !h->tr_xdot)) return fail(DEMCMC_ENOMEM, "trace buffers do not fit");
        if (h->tr_xdot) BE(be::dzero(h->tr_xdot, sizeof(double) * S * P));
        if (!h->block_on.empty()) {                              // sweep slots of unblocked iterations stay unused: read as zero
            BE(be::dzero(h->tr_theta, sizeof(double) * S * P * d)); BE(be::dzero(h->tr_w, sizeof(double) * S * P));
            BE(be::dzero(h->tr_adj, sizeof(double) * S * P)); BE(be::dzero(h->tr_acc, (size_t)S * P));
        }
        h->tr_sweeps = S;
    }
    be::dfree(h->d_mig_log); h->d_mig_log = nullptr; h->mig_log_iters = n_iter;
    h->last_mig_slots.assign((size_t)std::max<int64_t>(1, n_iter) * h->cfg.n_groups, -1);
    if (n_iter > 0) {
        h->d_mig_log = (int32_t *)be::dmalloc(sizeof(int32_t) * n_iter * MAX_MIG);
        if (!h->d_mig_log) return fail(DEMCMC_ENOMEM, "migration log");
        BE(be::dfill(h->d_mig_log, 0xFF, sizeof(int32_t) * n_iter * MAX_MIG));   // -1: a cycle this rank took no part in
    }
    return 0;
}

static void get_mig(const demcmc_handle *h, const RunCall &call, int64_t it, MigSchedule &out)
{
    const int Gt = h->cfg.n_groups;
    const demcmc_tape *tape = call.tape;
    out.migrate = false; out.n = 0; out.groups.clear(); out.u_pick.clear();
    if (Gt < 2) return;
    if (!tape) return plan_migration(h->cfg.seed, (uint32_t)(h->iter_offset + h->iters_done + it), Gt, h->cfg.alpha, out);
    out.n = tape->mig_n[it]; out.migrate = out.n > 0;
    for (int i = 0; i < out.n; ++i) { out.groups.push_back(tape->mig_groups[it * Gt + i]); out.u_pick.push_back(tape->mig_pick_u[it * Gt + i]); }
}
static bool in_burnin_at(const demcmc_handle *h, int64_t it) { return h->iter_offset + h->iters_done + it + 1 + h->cfg.n_initial <= h->cfg.burnin; }   // de.iter <= burnin
// native select_base reads the sweep-start weights: such a sweep starts from a complete state
static bool needs_snapshot(const demcmc_handle *h, const RunCall &call, int64_t it) { return !call.tape && h->cfg.proposal == DEMCMC_RANDOM_GAMMA && in_burnin_at(h, it); }
// blocking_on(de) (main.jl:137,162) of local iteration `it`
static bool blocking_at(const demcmc_handle *h, int64_t it)
{
    const int64_t a = h->iter_offset + h->iters_done + it;
    return h->B > 1 && (a >= (int64_t)h->block_on.size() || h->block_on[(size_t)a] != 0);
}

// the sweep contexts of a chunk, and the rows its sweeps write: the current state moves to the chunk's last row
static void fill_sweep_contexts(demcmc_handle *h, const RunCall &call, Chunk &ck)
{
    const int G = h->G_local, P = h->P, d = h->d, B = h->B;
    const TapeShard &ts = call.shard; const bool blocked = ck.blocked, ghist = call.ghist;
    const int64_t itg0 = h->iters_done + ck.it0;
    Row cur = cur_row(h);
    for (int s = 0; s < ck.n_sw; ++s) {
        // a chunk of blocked sweeps walks the blocks of consecutive iterations: sweep s is block (b0 + s) % B of
        // iteration it0 + (b0 + s) / B; an unblocked chunk holds one sweep per iteration
        const int b = blocked ? (ck.b0 + s) % B : 0;
        const int64_t it = ck.it0 + (blocked ? (ck.b0 + s) / B : s), itg = itg0 + (blocked ? (ck.b0 + s) / B : s);
        const bool last = !blocked || b == B - 1;             // this sweep completes its iteration
        const int64_t s_local = it * B + b;
        const bool inb = in_burnin_at(h, it);
        ck.basedep[s] = call.tape && h->cfg.proposal == DEMCMC_RANDOM_GAMMA && inb;
        // destination row: the history row of the iteration on its last block, else scratch
        // (thinning: only every k_store-th iteration has a history row; the others live in the scratch ring,
        // whose MAX_CHUNK + 2 rows keep every row of a chunk write-once)
        const bool stored = last && (itg + 1) % h->k_store == 0;
        const int64_t hist_row = h->n0 + (itg + 1) / h->k_store - 1;
        Row next;
        int next_scratch = -1;
        if (stored) next = row_of(h, true, hist_row);
        else {
            // never the row of an earlier sweep of this chunk: overlapped sweeps read each other's rows out of
            // order (a late update of sweep t still reads row t-1 while sweep t+3 is being written)
            next_scratch = h->scr_cursor = (h->scr_cursor + 1) % h->n_scratch;
            if (h->cur_hist < 0 && next_scratch == h->cur_scratch) next_scratch = h->scr_cursor = (h->scr_cursor + 1) % h->n_scratch;
            next = row_of(h, false, next_scratch);
        }
        SweepCtx &ctx = ck.u.h_ctx[s];
        memset(&ctx, 0, sizeof ctx);
        ctx.sweep = (uint32_t)((h->iter_offset + itg) * B + b); ctx.block = blocked ? b : -1; ctx.in_burnin = inb; ctx.replay = call.tape != nullptr;
        ctx.exact_base = call.tape != nullptr;
        ctx.cur_theta = cur.theta; ctx.cur_w = cur.w; ctx.cur_id = cur.id;
        ctx.next_theta = next.theta; ctx.next_w = next.w; ctx.next_id = next.id; ctx.next_acc = next.acc;
        ctx.mutate = ck.u.d_mut + (size_t)s * G;
        ctx.plan = (call.tape || !h->plan_recs) ? nullptr : h->plan_recs + (size_t)s * P;
        if (call.tape) {
            ctx.t_kind = ts.t_kind + (size_t)s_local * P; ctx.t_idx = ts.t_idx + (size_t)s_local * P * 3;
            ctx.t_g1 = ts.t_g1 + (size_t)s_local * P; ctx.t_g2 = ts.t_g2 + (size_t)s_local * P; ctx.t_uacc = ts.t_uacc + (size_t)s_local * P;
            ctx.t_noise = ts.t_noise + (size_t)s_local * P * d; ctx.t_keep = ts.t_keep ? ts.t_keep + (size_t)s_local * P * d : nullptr;
            ctx.t_idx_row = ts.t_idx_row ? ts.t_idx_row + (size_t)s_local * P * 3 : nullptr;
        }
        ctx.prop_theta = h->prop_theta; ctx.prop_prior = h->prop_prior; ctx.prop_adj = h->prop_adj; ctx.prop_inb = h->prop_inb; ctx.prop_msq = h->prop_msq;
        ctx.ll_part = h->ll_part; ctx.ll_acc = h->ll_acc; ctx.ll_q = h->ll_q;
        ctx.base_cw = h->base_cw; ctx.base_tot = h->base_tot;
        // resample: donors are (row, id) cells of the rows stored before this iteration (crossover.jl:115)
        ctx.hist_theta = ghist ? h->ghist_theta : h->hist_theta; ctx.hist_pos = ghist ? h->ghist_pos : h->hist_pos; ctx.donor_rows = stored_rows(h, itg);
        ctx.next_pos = (stored && h->hist_pos && !ghist) ? h->hist_pos + (size_t)hist_row * P : nullptr;
        if (h->tr_sweeps) {
            ctx.tr_theta = h->tr_theta + (size_t)s_local * P * d; ctx.tr_w = h->tr_w + (size_t)s_local * P;
            ctx.tr_adj = h->tr_adj + (size_t)s_local * P; ctx.tr_acc = h->tr_acc + (size_t)s_local * P;
            ctx.tr_xdot = h->tr_xdot ? h->tr_xdot + (size_t)s_local * P : nullptr;
        }
        if (stored) { h->cur_hist = hist_row; }
        else { h->cur_hist = -1; h->cur_scratch = next_scratch; }
        cur = next;
    }
}

// Lanes: the groups split into independent sets (groups never read each other between migrations), each planned on
// its own and launched as its own kernel chain on its own stream, so one lane's likelihood kernel runs while the other
// lane proposes / accepts.
static int plan_lanes(demcmc_handle *h, RunCall &call, Chunk &ck)
{
    const demcmc_config &cfg = h->cfg; const bool blocked = ck.blocked; Upload &u = ck.u;
    const int Np = cfg.Np, G = h->G_local, P = h->P, B = h->B, n_lanes = call.n_lanes;
    static const int shape_mod = [] { const char *e = getenv("DEMCMC_SHAPE"); return std::max(0, e ? atoi(e) : 8); }();   // 0 = off, else the modulus (A/B runs)
    // levels of at most 112 updates (14 octets) for the persistent chunk kernel: measured on configs[1] against
    // no cap / 64 / 96 / 104 / 120 / 128: 2.86 M updates/s against 2.83 / 2.64 / 2.75 / 2.82 / 2.80 / 2.83
    static const int level_cap = [] { const char *e = getenv("DEMCMC_LEVEL_CAP"); return e ? std::max(0, atoi(e)) : 112; }();
    ck.lane_off[0] = 0;
    for (int ln = 0; ln < n_lanes; ++ln) {
        const int g0 = (ln * G + n_lanes - 1) / n_lanes, g1 = ((ln + 1) * G + n_lanes - 1) / n_lanes;   // contiguous sets of groups
        PlanInput pin;
        pin.seed = cfg.seed; pin.Np = Np; pin.G_local = g1 - g0; pin.group_begin = cfg.group_begin + g0; pin.G_total = cfg.n_groups;
        pin.pos_offset = g0 * Np; pin.P_stride = blocked ? P : P * B;   // consecutive sweeps of an unblocked chunk are consecutive iterations;
                                                                        // those of a blocked one are consecutive blocks (adjacent in the tape)
        pin.sweep_stride = blocked ? 1 : B;
        pin.shape_octets = is_ssd(h->dmodel.kind) ? shape_mod : 0;
        pin.level_cap = call.persist_lanes ? level_cap : 0;
        pin.proposal = cfg.proposal; pin.beta = cfg.beta; pin.theta_snooker = cfg.theta_snooker; pin.resample = cfg.donors != 0;
        const int64_t s_first = ck.it0 * B + (blocked ? ck.b0 : 0);
        pin.t_kind = call.tape ? call.shard.hk.data() + (size_t)s_first * P : nullptr;       // a chunk of several sweeps is unblocked: its sweeps are P_stride apart in the tape
        pin.t_idx = call.tape ? call.shard.hi.data() + (size_t)s_first * P * 3 : nullptr;
        ChunkPlan &pl = call.plans[ln];
        { HostTimer timer{ call.host_plan_s }; plan_chunk(pin, (uint32_t)((h->iter_offset + h->iters_done + ck.it0) * B + (blocked ? ck.b0 : 0)), ck.n_sw, ck.basedep, pl); }
        memcpy(u.h_order + ck.lane_off[ln], pl.order.data(), sizeof(int32_t) * pl.order.size());
        ck.lane_off[ln + 1] = ck.lane_off[ln] + (int32_t)pl.order.size();
        for (int s2 = 0; s2 < ck.n_sw; ++s2)
            for (int g = g0; g < g1; ++g) u.h_mut[(size_t)s2 * G + g] = pl.mutate[(size_t)s2 * (g1 - g0) + (g - g0)];
    }
    BE(be::h2d(u.d_blk, u.h_blk, u.off_order + sizeof(int32_t) * (size_t)ck.n_sw * P));   // contexts, flags and entries in one copy
    BE(be::event_record(u.copied));
    u.armed = true;
    if (!call.tape && h->plan_recs) BE(be::launch_plan(h->dcfg, u.d_ctx, ck.n_sw));     // every state-independent draw of the chunk, one launch
    return 0;
}

// Launches a planned chunk: the whole chunk in one persistent launch where that kernel takes it, else every level in
// one single-CTA launch where that kernel takes it, else level by level.
static int launch_chunk(demcmc_handle *h, RunCall &call, const Chunk &ck)
{
    const Upload &u = ck.u; const ChunkPlan *plans = call.plans; const int n_lanes = call.n_lanes;
    if (needs_snapshot(h, call, ck.it0) && std::count(u.h_mut, u.h_mut + h->G_local, 0) > 0)    // n_sw == 1 here; a group crosses over
        BE(be::launch_base_prep(h->dcfg, u.h_ctx[0].cur_w, h->base_th, h->base_cw, h->base_tot));
    int max_levels = 0;
    for (int ln = 0; ln < n_lanes; ++ln) max_levels = std::max(max_levels, plans[ln].n_levels);
    // ---- the persistent path: the whole chunk in one launch (MVN / hierarchical) ---------------
    // levels of the lanes alternate; a level's proposals wait for the previous level of its lane
    if (call.persist_lanes) {
        std::vector<int32_t> off, cnt, dep;
        int last[be::MAX_LANES];                                 // the last level of each lane so far
        std::fill_n(last, be::MAX_LANES, -1);
        for (int l = 0; l < max_levels; ++l)
            for (int ln = 0; ln < n_lanes; ++ln) {
                const ChunkPlan &pl = plans[ln];
                if (l >= pl.n_levels || pl.level_off[l + 1] == pl.level_off[l]) continue;
                off.push_back(ck.lane_off[ln] + pl.level_off[l]);
                cnt.push_back(pl.level_off[l + 1] - pl.level_off[l]);
                dep.push_back(last[ln]);
                last[ln] = (int)off.size() - 1;
            }
        const bool tl = h->time_loglik && call.tev_ll0 + 2 * call.tev_ll + 1 < h->tev.size();
        if (tl) BE(be::event_record(h->tev[call.tev_ll0 + 2 * call.tev_ll]));
        const int rc = off.empty() ? 1 : be::launch_chunk_persist(h->dcfg, h->dmodel, u.d_order, u.d_ctx, off.data(), cnt.data(), dep.data(),
                                                                  (int)off.size(), n_lanes > 1 ? 1 : 0, h->ll_acc, std::max(2, n_lanes));
        if (rc < 0) return fail(DEMCMC_ECUDA, "chunk launch: %s", be::last_error());
        if (rc == 0) {
            if (tl) { BE(be::event_record(h->tev[call.tev_ll0 + 2 * call.tev_ll + 1])); ++call.tev_ll; }
            call.n_levels += (int64_t)off.size();
            ++h->ctr.persistent_chunks;
            return 0;
        }
    }
    // ---- a population of a few warps (the reference's own examples): every level of the chunk in one single-CTA launch
    if (n_lanes == 1 && !h->time_loglik && !call.skip_stream) {
        const ChunkPlan &pl = plans[0];
        const int rc = be::launch_chunk_small(h->dcfg, h->dmodel, u.d_order, u.d_ctx, pl.level_off.data(), pl.n_levels);
        if (rc < 0) return fail(DEMCMC_ECUDA, "chunk launch: %s", be::last_error());
        if (rc == 0) { call.n_levels += pl.n_levels; return 0; }
    }
    BE(be::lane_fork(n_lanes));
    int rc_launch = 0;
    for (int l = 0; l < max_levels && !rc_launch; ++l)
        for (int ln = 0; ln < n_lanes && !rc_launch; ++ln) {
            const ChunkPlan &pl = plans[ln];
            if (l >= pl.n_levels || pl.level_off[l + 1] == pl.level_off[l]) continue;
            const Level lv = { u.d_order + ck.lane_off[ln] + pl.level_off[l], pl.level_off[l + 1] - pl.level_off[l], u.d_ctx };
            be::set_lane(ln);
            const bool tl = h->time_loglik && call.tev_ll0 + 2 * call.tev_ll + 1 < h->tev.size();
            if (!tl) {
                const int fused = be::launch_level_fused(h->dcfg, h->dmodel, lv);
                if (fused < 0) { rc_launch = 1; break; }
                if (fused == 0) { ++call.n_levels; continue; }
            }
            if (be::launch_propose(h->dcfg, h->dmodel, lv) ||
                (tl && be::event_record(h->tev[call.tev_ll0 + 2 * call.tev_ll])) ||
                (!call.skip_stream && be::launch_loglik(h->dcfg, h->dmodel, h->prop_theta, lv, h->ll_part, h->ll_acc)) ||
                (tl && be::event_record(h->tev[call.tev_ll0 + 2 * call.tev_ll + 1])) ||
                be::launch_accept(h->dcfg, h->dmodel, lv)) rc_launch = 1;
            if (tl) ++call.tev_ll;
            ++call.n_levels;
        }
    be::set_lane(0);
    if (rc_launch) return fail(DEMCMC_ECUDA, "level launch: %s", be::last_error());
    BE(be::lane_join(n_lanes));
    return 0;
}

// ---- migration! (main.jl:85, migration.jl:11-19) before local iteration `it`, on the current row, in place --------
static int migrate(demcmc_handle *h, RunCall &call, int64_t it)
{
    const int Gt = h->cfg.n_groups, P = h->P, d = h->d;
    MigSchedule ms;
    get_mig(h, call, it, ms);
    if (!ms.migrate) return 0;
    Row cur = cur_row(h);
    if (ms.n < 2 || ms.n > Gt) return fail(DEMCMC_EINVAL, "migration with %d groups", ms.n);
    MigArgs a;
    memset(&a, 0, sizeof a);
    a.n = ms.n;
    bool cross = false, any_local = false;
    std::vector<int> src(ms.n), dst(ms.n);
    for (int i = 0; i < ms.n; ++i) {
        a.groups[i] = ms.groups[i]; a.u_pick[i] = ms.u_pick[i];
        if (a.groups[i] < 0 || a.groups[i] >= Gt) return fail(DEMCMC_EINVAL, "migration group out of range");
        dst[i] = h->group_owner[ms.groups[i]];
        src[i] = h->group_owner[ms.groups[(i + ms.n - 1) % ms.n]];
        a.src_rank[i] = (int8_t)src[i]; a.dst_rank[i] = (int8_t)dst[i];
        cross |= src[i] != dst[i];
        any_local |= dst[i] == h->rank;
    }
    // a cycle that spans ranks is one mailbox EVENT on every rank (the schedule is the same everywhere): slot
    // seq % depth, published under the tag seq + 1; before a slot is used again every rank must have consumed it
    const bool use_mbox = cross && h->mbox_on;
    if (cross) ++h->ctr.cross_migrations;
    if (use_mbox) ++h->ctr.mailbox_events;
    int mb_slot = 0;
    unsigned long long mb_tag = 0;
    if (use_mbox) {
        uint64_t &seq = *h->mbox_seq_p;
        if (seq > 0 && seq % (uint64_t)h->mbox.depth == 0 && h->mbox_barrier)
            if (h->mbox_barrier()) return fail(DEMCMC_ECOMM, "mailbox barrier: %s", be::last_error());
        mb_slot = (int)(seq % (uint64_t)h->mbox.depth);
        mb_tag = seq + 1;
        ++seq;
    }
    if (any_local || cross) {
        int32_t *picks = h->d_mig_log + it * MAX_MIG;
        BE(be::launch_mig_pick(h->dcfg, a, cur.w, picks));
        BE(be::launch_mig_gather(h->dcfg, a, picks, cur.theta, cur.w, cur.id, cur.acc, h->d_stage));
        const double *incoming = h->d_stage;
        if (use_mbox) {
            BE(be::launch_mig_push(h->dcfg, a, h->d_stage, h->peers, h->mbox, h->rank, mb_slot, mb_tag));
        } else if (cross) {
            if (!h->comm) return fail(DEMCMC_ECOMM, "migration crosses ranks but demcmc_comm_init was not called");
            BE(be::d2d(h->d_stage_recv, h->d_stage, sizeof(double) * ms.n * (d + 3)));
            if (be::comm_exchange(h->comm, h->rank, ms.n, src.data(), dst.data(), h->d_stage, h->d_stage_recv, d + 3)) return fail(DEMCMC_ECOMM, "%s", be::last_error());
            incoming = h->d_stage_recv;
        }
        BE(be::launch_mig_scatter(h->dcfg, a, picks, incoming, cur.theta, cur.w, cur.id, cur.acc,
                                  (h->hist_pos && h->cur_hist >= 0 && !call.ghist) ? h->hist_pos + (size_t)h->cur_hist * P : nullptr,
                                  use_mbox ? &h->mbox : nullptr, h->rank, mb_slot, mb_tag));
    }
    // the migration edited a stored row: refresh its replicated copy (collective: every rank, the
    // schedule is the same everywhere)
    if (call.ghist && h->cur_hist >= 0) if (int rc = gather_row(h, h->cur_hist)) return rc;
    call.mig_events.emplace_back(it, ms.n);
    return 0;
}

// Sweeps in the chunk that starts at local iteration `it`.  Consecutive iterations without a migration, without a
// sweep-start snapshot and in the same blocking mode overlap on the device: they are planned as one chunk (planner.h).
// 1 for a blocked iteration: its blocks run as chunks of one sweep each.
static int chunk_length(demcmc_handle *h, RunCall &call, int64_t it, bool blocked)
{
    const int B = h->B; int64_t max_it;                          // iterations the chunk may hold
    if (blocked) {
        // blocking (main.jl:174-179): every block is one sweep.  Consecutive block sweeps -- the blocks of this
        // iteration and of the blocked iterations that follow it without a migration in between -- overlap on the
        // device like the sweeps of unblocked iterations do (the tail levels of one sweep share launches with the
        // head levels of the next).  A sweep whose select_base needs the sweep-start weights, and DE-MCz donors
        // (rows of earlier sweeps), keep one sweep per chunk.
        if (needs_snapshot(h, call, it) || h->cfg.donors || h->max_chunk <= 1) return 1;
        const int cap_sweeps = (int)std::min<int64_t>(h->max_chunk, (int64_t)4 << std::min<int64_t>(call.chunks_this_call, 8));
        max_it = std::max(cap_sweeps, B) / B;
    } else {
        // slow start: the device idles while the host plans the first chunk of a call (49 ms for 16
        // sweeps of 32768 particles), so the first chunks are short -- 2, 4, 8 sweeps -- and the long
        // ones are planned while the device is busy with their predecessors
        static const int first_chunk = [] { const char *e = getenv("DEMCMC_FIRST_CHUNK"); return e ? std::max(1, atoi(e)) : 4; }();     // 4, 8, 16 sweeps: measured against 2, 4, 8, 16 at 20 steps: +1.4 %
        // ... doubling from chunk to chunk; four-fold where a sweep is heavy on the device next to its planning (>= 2e6
        // observation x dimension products per particle: planning 16 sweeps of configs[1] takes 0.6 ms, the 4 sweeps it hides
        // behind 1.5 ms), so that a 20-iteration call is 4 + 16 sweeps instead of 4 + 8 + 8
        static const int growth_env = [] { const char *e = getenv("DEMCMC_CHUNK_GROWTH"); return e ? std::max(0, atoi(e)) : 0; }();
        const bool heavy = (double)h->dmodel.n_obs * (double)std::max(1, (int)h->dmodel.n_dim) >= 2e6;
        const int shift = growth_env ? growth_env : (heavy ? 2 : 1);
        const int chunk_cap = (int)std::min<int64_t>(h->max_chunk, (int64_t)first_chunk << std::min<int64_t>(shift * call.chunks_this_call, 8));
        // resample reads rows of earlier sweeps: one sweep per chunk
        max_it = (needs_snapshot(h, call, it) || h->max_chunk <= 1 || h->cfg.donors) ? 1 : chunk_cap;
    }
    ++call.chunks_this_call;
    int n = 1; MigSchedule m2;
    while (it + n < call.n_iter && n < max_it) {
        get_mig(h, call, it + n, m2);
        if (m2.migrate || needs_snapshot(h, call, it + n) || blocking_at(h, it + n) != blocked) break;
        ++n;
    }
    return !blocked ? n : n * B > MAX_CHUNK ? 1 : n * B;        // more blocks than a chunk holds: one sweep per chunk
}

static int run_impl(demcmc_handle *h, const demcmc_tape *tape, int64_t n_iter)
{
    if (!h || n_iter < 0) return fail(DEMCMC_EINVAL, "bad argument");
    if (!h->has_model || !h->has_state) return fail(DEMCMC_ESTATE, "set_model and set_state must come before run");
    BE(be::set_device(h->cfg.device));
    const demcmc_config &cfg = h->cfg; const int Gt = cfg.n_groups, G = h->G_local, P = h->P, B = h->B;
    if (h->n0 > 0 && !h->has_history) return fail(DEMCMC_ESTATE, "n_initial > 0: demcmc_set_history must come before run");
    if (cfg.donors && G != Gt && h->n_ranks <= 1) return fail(DEMCMC_ESTATE, "sample = resample on a sharded job reads the history of every particle id: demcmc_comm_init must come first");
    RunCall call;
    call.tape = tape; call.n_iter = n_iter; call.S = n_iter * B; call.ghist = cfg.donors && h->n_ranks > 1;
    h->dcfg.P_hist = call.ghist ? (int32_t)((int64_t)Gt * cfg.Np) : (int32_t)P;
    if (cfg.donors && h->iter_offset > 0) return fail(DEMCMC_EUNSUPPORTED, "sample = resample draws donors from the rows of earlier iterations: a resumed handle does not hold them");
    if (int rc = grow_history(h, stored_rows(h, h->iters_done + n_iter))) return rc;
    if (tape) if (int rc = load_tape(h, tape, n_iter, call.shard)) return rc;
    if (int rc = reset_call_buffers(h, call)) return rc;

    const int64_t launches0 = be::launch_count();
    call.tev_ll0 = h->flush_bytes ? 2 * (size_t)n_iter : 0;
    const size_t tev_need = call.tev_ll0 + (h->time_loglik ? 2 * (size_t)call.S * 64 : 0);
    while (h->tev.size() < tev_need) { void *e = be::tevent_create(); if (!e) return fail(DEMCMC_ECUDA, "event pool: %s", be::last_error()); h->tev.push_back(e); }
    BE(be::timer_start());
    // the persistent chunk kernel alternates the levels of two lanes; the level-by-level path runs the handle's lanes
    // (default 1) as concurrent kernel chains
    call.skip_stream = h->suffstat && is_ssd(h->dmodel.kind);    // B == 0 analytically: propose -> accept, nothing streamed
    call.persist_lanes = call.skip_stream ? 0 : be::chunk_persist_lanes(h->dcfg, h->dmodel);
    call.n_lanes = call.persist_lanes ? call.persist_lanes : std::max(1, std::min(h->n_lanes, G));

    for (int64_t it = 0; it < n_iter;) {
        // measurement mode: one timed segment = the migration (with its NCCL exchange) plus the chunk(s)
        // that follow it; the L2 flush in front of the segment is outside the bracket
        if (h->flush_bytes) { BE(be::dfill(h->flush_buf, (int)(call.tev_chunks & 1), (size_t)h->flush_bytes)); BE(be::event_record(h->tev[2 * call.tev_chunks])); }
        if (int rc = migrate(h, call, it)) return rc;
        // ---- update! (main.jl:161-167) -------------------------------------------------------------
        const bool blocked = blocking_at(h, it);
        const int n_sw = chunk_length(h, call, it, blocked);
        const int n_chunks = blocked && n_sw == 1 ? B : 1;
        for (int c = 0; c < n_chunks; ++c) {
            call.sweeps_run += n_sw;
            HostTimer timer{ call.host_chunk_s };
            Chunk ck{ it, c, n_sw, blocked, h->ring[h->ring_use % demcmc_handle::RING] };
            if (ck.u.armed) BE(be::event_wait(ck.u.copied));   // the pinned slot is free once its copies ran
            h->ring_use++;
            fill_sweep_contexts(h, call, ck);
            if (int rc = plan_lanes(h, call, ck)) return rc;
            if (int rc = launch_chunk(h, call, ck)) return rc;
        }
        if (call.ghist && h->cur_hist >= 0) if (int rc = gather_row(h, h->cur_hist)) return rc;     // resample: one sweep per chunk
        if (h->flush_bytes) { BE(be::event_record(h->tev[2 * call.tev_chunks + 1])); ++call.tev_chunks; }
        it += blocked ? n_chunks * n_sw / B : n_sw;
    }
    double ms_dev = 0.0;
    BE(be::timer_stop(&ms_dev));
    BE(be::sync());
    if (h->flush_bytes) {                                   // sum of the per-segment times (migration + chunk), flushes excluded
        ms_dev = 0.0;
        for (size_t c = 0; c < call.tev_chunks; ++c) { double t = 0.0; BE(be::tevent_elapsed(h->tev[2 * c], h->tev[2 * c + 1], &t)); ms_dev += t; }
    }
    double ms_ll = 0.0;
    for (size_t i = 0; i < call.tev_ll; ++i) { double t = 0.0; BE(be::tevent_elapsed(h->tev[call.tev_ll0 + 2 * i], h->tev[call.tev_ll0 + 2 * i + 1], &t)); ms_ll += t; }
    h->ctr.loglike_ms = ms_ll;
    for (auto &ev : call.mig_events)                        // migration log -> host
        BE(be::d2h(h->last_mig_slots.data() + ev.first * Gt, h->d_mig_log + ev.first * MAX_MIG, sizeof(int32_t) * ev.second));
    h->iters_done += n_iter;
    if (host_profile()) fprintf(stderr, "[demcmc host] %lld iterations: chunks %.3f ms on the host (planner %.3f ms), %lld levels\n", (long long)n_iter, call.host_chunk_s * 1e3, call.host_plan_s * 1e3, (long long)call.n_levels);
    h->ctr.iterations += n_iter; h->ctr.sweeps += call.sweeps_run; h->ctr.particle_updates += call.sweeps_run * P; h->ctr.loglike_evals += call.sweeps_run * P;
    h->ctr.kernel_launches += be::launch_count() - launches0; h->ctr.levels += call.n_levels; h->ctr.device_ms = ms_dev;
    return 0;
}

// a multi-device handle: one host thread per device, each running the loop of its own groups; the devices meet only in
// the migration mailboxes (and in a host barrier when a mailbox slot comes up for reuse)
static int multi_run(demcmc_handle *h, const demcmc_tape *tape, int64_t n_iter)
{
    if (n_iter < 0) return fail(DEMCMC_EINVAL, "bad argument");
    // sample = resample: the devices store into each other's replicated history, so every copy has its final address
    // before any device starts (run_impl then finds the capacity in place)
    if (h->cfg.donors)
        if (const int rc = for_kids(h, [&](demcmc_handle *k, int) {
                if (be::set_device(k->cfg.device)) return fail(DEMCMC_ECUDA, "%s", be::last_error());
                if (int r = grow_history(k, stored_rows(k, k->iters_done + n_iter))) return r;
                return be::sync() ? fail(DEMCMC_ECUDA, "%s", be::last_error()) : 0;
            }, false)) return rc;
    h->multi->barrier.reset();
    const int rc = for_kids(h, [&](demcmc_handle *k, int) {
        const int r = run_impl(k, tape, n_iter);
        if (r) h->multi->barrier.abort();                  // the peers must not wait for this device at a host barrier
        return r;
    });
    if (!rc) h->iters_done += n_iter;
    return rc;
}
int demcmc_run(demcmc_handle *h, int64_t n_iter) { return (h && h->multi) ? multi_run(h, nullptr, n_iter) : run_impl(h, nullptr, n_iter); }
int demcmc_replay(demcmc_handle *h, const demcmc_tape *tape, int64_t n_iter)
{
    if (!tape) return fail(DEMCMC_EINVAL, "null tape");
    return (h && h->multi) ? multi_run(h, tape, n_iter) : run_impl(h, tape, n_iter);
}

static int history_out(demcmc_handle *h, double *samples, double *lp, uint8_t *accept, int64_t n_rows)
{
    if (!h) return fail(DEMCMC_EINVAL, "null handle");
    if (h->multi) return multi_history_out(h, samples, lp, accept, n_rows);
    if (n_rows != stored_rows(h)) return fail(DEMCMC_EINVAL, "n_rows %lld != the %lld stored rows (iterations run / store_every + n_initial)", (long long)n_rows, (long long)stored_rows(h));
    if (h->n_ranks > 1) return fail(DEMCMC_EUNSUPPORTED, "by-id history of a sharded job: gather demcmc_get_history_by_slot on the host");
    BE(be::set_device(h->cfg.device));
    const size_t P = h->P, d = h->d;
    const int64_t n0 = h->cfg.n_initial;
    double *ds = nullptr, *dl = nullptr; uint8_t *da = nullptr;
    int rc = 0;
    if (samples) ds = (double *)be::dmalloc(sizeof(double) * std::max<size_t>(1, n_rows * P * d));
    if (lp) dl = (double *)be::dmalloc(sizeof(double) * std::max<size_t>(1, n_rows * P));
    const bool lp_written = h->cfg.update == DEMCMC_UPDATE_MH;     // maximize!/minimize! leave Particle.lp at 0.0
    if (accept) da = (uint8_t *)be::dmalloc(std::max<size_t>(1, n_rows * P));
    if ((samples && !ds) || (lp && !dl) || (accept && !da)) rc = fail(DEMCMC_ENOMEM, "output staging does not fit on the device");
    if (!rc && n_rows > 0) {
        if (ds && be::dzero(ds, sizeof(double) * n_rows * P * d)) rc = DEMCMC_ECUDA;
        if (dl && be::dzero(dl, sizeof(double) * n_rows * P)) rc = DEMCMC_ECUDA;
        if (da && be::dzero(da, n_rows * P)) rc = DEMCMC_ECUDA;
        if (!rc && stored_rows(h) > 0 && (n0 == 0 || h->has_history) &&
            be::launch_history_by_id(h->hist_theta, h->hist_w, h->hist_acc, h->hist_id, stored_rows(h), 0, n_rows, (int32_t)P, (int32_t)d,
                                     h->cfg.group_begin * h->cfg.Np, ds, lp_written ? dl : nullptr, da)) rc = DEMCMC_ECUDA;
        if (!rc && ds && be::d2h(samples, ds, sizeof(double) * n_rows * P * d)) rc = DEMCMC_ECUDA;
        if (!rc && dl && be::d2h(lp, dl, sizeof(double) * n_rows * P)) rc = DEMCMC_ECUDA;
        if (!rc && da && be::d2h(accept, da, n_rows * P)) rc = DEMCMC_ECUDA;
        if (rc == DEMCMC_ECUDA) fail(rc, "history gather: %s", be::last_error());
    }
    be::dfree(ds); be::dfree(dl); be::dfree(da);
    return rc;
}

int demcmc_get_samples(demcmc_handle *h, double *out, int64_t n_rows) { return out ? history_out(h, out, nullptr, nullptr, n_rows) : fail(DEMCMC_EINVAL, "null out"); }
int demcmc_get_accept(demcmc_handle *h, uint8_t *out, int64_t n_rows) { return out ? history_out(h, nullptr, nullptr, out, n_rows) : fail(DEMCMC_EINVAL, "null out"); }
int demcmc_get_lp(demcmc_handle *h, double *out, int64_t n_rows) { return out ? history_out(h, nullptr, out, nullptr, n_rows) : fail(DEMCMC_EINVAL, "null out"); }

int demcmc_get_moments(demcmc_handle *h, int64_t row0, int64_t n_rows, int64_t *count, double *mean, double *m2)
{
    if (!h || !count || !mean || !m2) return fail(DEMCMC_EINVAL, "null argument");
    if (h->multi) return multi_get_moments(h, row0, n_rows, count, mean, m2);
    if (row0 < 0 || n_rows < 0 || row0 + n_rows > stored_rows(h)) return fail(DEMCMC_EINVAL, "row range [%lld, %lld) outside the %lld stored rows", (long long)row0, (long long)(row0 + n_rows), (long long)stored_rows(h));
    BE(be::set_device(h->cfg.device));
    const size_t P = h->P, d = h->d;
    *count = n_rows * (int64_t)P;
    if (n_rows == 0) { for (size_t k = 0; k < d; ++k) { mean[k] = 0.0; m2[k] = 0.0; } return 0; }
    double *out = (double *)be::dmalloc(sizeof(double) * 2 * d);
    if (!out) return fail(DEMCMC_ENOMEM, "moments staging");
    int rc = 0;
    if (be::launch_moments(h->hist_theta + (size_t)row0 * P * d, n_rows * (int64_t)P, (int32_t)d, out, out + d) ||
        be::d2h(mean, out, sizeof(double) * d) || be::d2h(m2, out + d, sizeof(double) * d))
        rc = fail(DEMCMC_ECUDA, "moments: %s", be::last_error());
    be::dfree(out);
    return rc;
}

// split-R-hat and ESS from the aggregates of launch_diag_aggregates, summed over the shards (m = split chains in all).
// head[k] = the three variance sums, acov[k] = the chain-summed autocovariances of the lags computed so far; returns
// false when some parameter's Geyer sequence is still positive at the last lag available and lags remain (< nh)
static bool diag_finish(const std::vector<std::array<double, 3>> &head, const std::vector<std::vector<double>> &acov, int64_t nh, int64_t m, double *rhat, double *ess)
{
    const double n = (double)nh, M = (double)m;
    bool done = true;
    for (size_t k = 0; k < head.size(); ++k) {
        const double *a = acov[k].data();
        const int64_t n_lag = (int64_t)acov[k].size();
        const double W = head[k][0] / M;                                  // mean within-chain variance
        const double var_means = M > 1 ? (head[k][2] - head[k][1] * head[k][1] / M) / (M - 1.0) : 0.0;
        const double var_plus = W * (n - 1.0) / n + var_means;           // B / n = var of the chain means
        if (rhat) rhat[k] = W > 0.0 ? sqrt(var_plus / W) : NAN;
        if (!ess) continue;
        if (!(var_plus > 0.0)) { ess[k] = NAN; continue; }
        auto rho = [&](int64_t t) { return t == 0 ? 1.0 : 1.0 - (W - a[t] / M) / var_plus; };
        double tau = -1.0, prev = INFINITY;
        bool ended = false;
        for (int64_t t = 0; t + 1 < n_lag; t += 2) {                      // Geyer's initial positive, monotone sequence
            double pair = rho(t) + rho(t + 1);
            if (pair < 0.0) { ended = true; break; }
            pair = std::min(pair, prev);
            prev = pair;
            tau += 2.0 * pair;
        }
        if (!ended && n_lag < nh) done = false;
        tau = std::max(tau, 1.0 / log10(std::max(n * M, 10.0)));
        ess[k] = n * M / tau;
    }
    return done;
}

int demcmc_get_diagnostics(demcmc_handle *h, int64_t row0, int64_t n_rows, double *rhat, double *ess)
{
    if (!h || (!rhat && !ess)) return fail(DEMCMC_EINVAL, "null argument");
    demcmc_handle *h0 = h->multi ? h->kids[0] : h;
    if (row0 < 0 || n_rows < 4 || row0 + n_rows > stored_rows(h0)) return fail(DEMCMC_EINVAL, "row range [%lld, %lld) outside the %lld stored rows (at least 4 rows)", (long long)row0, (long long)(row0 + n_rows), (long long)stored_rows(h0));
    const int64_t nh = n_rows / 2;
    if (nh > be::diag_max_half()) return fail(DEMCMC_EUNSUPPORTED, "diagnostics over more than %d stored rows per call: thin the run or pass a sub-range", 2 * be::diag_max_half());
    // the autocovariances come in batches of lags (an even number: Geyer's sequence sums pairs); a batch is computed only
    // while some parameter's sequence is still positive at the last lag of the one before it
    // (DEMCMC_DIAG_LAGS: test switch, a smaller batch so that short chains walk through several of them)
    const char *lag_env = getenv("DEMCMC_DIAG_LAGS");
    const int d = h->d, lag_step = std::max(2, std::min(be::diag_max_lags(), lag_env ? atoi(lag_env) : be::diag_max_lags()) & ~1), n_lag = (int)std::min<int64_t>(nh, lag_step);
    const size_t na = (size_t)d * (3 + n_lag);
    std::vector<demcmc_handle *> leaves = h->multi ? h->kids : std::vector<demcmc_handle *>{ h };
    const int32_t Pt = (int32_t)h->P, id_base = h->multi ? 0 : h->cfg.group_begin * h->cfg.Np;
    // ids migrate between the shards of a job: every shard marks, in ONE map on the first device, where the ids it holds
    // sit at every row; the first device then gathers every chain through the map (peer access) and reduces
    BE(be::set_device(h0->cfg.device));
    int32_t *pos = (int32_t *)be::dmalloc_shared(sizeof(int32_t) * (size_t)n_rows * Pt);
    double *agg = (double *)be::dmalloc(sizeof(double) * na);
    std::vector<double> total(na);
    int rc = (!pos || !agg) ? fail(DEMCMC_ENOMEM, "diagnostics staging") : 0;
    DiagShards sh;
    memset(&sh, 0, sizeof sh);
    sh.n = (int32_t)leaves.size(); sh.P_local = (int32_t)h0->P;
    for (size_t i = 0; i < leaves.size() && !rc; ++i) {
        demcmc_handle *k = leaves[i];
        sh.theta[i] = k->hist_theta;
        if (be::set_device(k->cfg.device) ||
            be::launch_diag_pos(k->hist_id, row0, n_rows, (int32_t)k->P, id_base, Pt, h->multi ? k->cfg.group_begin * k->cfg.Np : 0, pos) || be::sync())
            rc = fail(DEMCMC_ECUDA, "diagnostics: %s", be::last_error());
    }
    std::vector<std::array<double, 3>> head(d);
    std::vector<std::vector<double>> acov(d);
    for (int64_t lag0 = 0; lag0 < nh && !rc; lag0 += lag_step) {
        const int nl = (int)std::min<int64_t>(lag_step, nh - lag0);
        if (be::set_device(h0->cfg.device) || be::launch_diag_aggregates(sh, pos, row0, n_rows, Pt, d, (int32_t)lag0, nl, agg) ||
            be::d2h(total.data(), agg, sizeof(double) * (size_t)d * (3 + nl))) { rc = fail(DEMCMC_ECUDA, "diagnostics: %s", be::last_error()); break; }
        for (int k = 0; k < d; ++k) {
            const double *a = total.data() + (size_t)k * (3 + nl);
            if (lag0 == 0) head[k] = { a[0], a[1], a[2] };
            acov[k].insert(acov[k].end(), a + 3, a + 3 + nl);
        }
        if (diag_finish(head, acov, nh, 2 * (int64_t)Pt, rhat, ess) || !ess) break;
    }
    be::set_device(h0->cfg.device);
    be::dfree_shared(pos); be::dfree(agg);
    return rc;
}

int demcmc_get_chains(demcmc_handle *h, int64_t row0, int64_t n_rows, double *out)
{
    if (!h || !out) return fail(DEMCMC_EINVAL, "null argument");
    if (h->multi) return multi_get_chains(h, row0, n_rows, out);
    if (row0 < 0 || n_rows < 0 || row0 + n_rows > stored_rows(h)) return fail(DEMCMC_EINVAL, "row range [%lld, %lld) outside the %lld stored rows", (long long)row0, (long long)(row0 + n_rows), (long long)stored_rows(h));
    if (h->n_ranks > 1) return fail(DEMCMC_EUNSUPPORTED, "chains of a sharded job: gather demcmc_get_history_by_slot on the host");
    if (!h->has_state) return fail(DEMCMC_ESTATE, "no state");
    BE(be::set_device(h->cfg.device));
    if (n_rows == 0) return 0;
    const size_t P = h->P, d = h->d, n = (size_t)n_rows * P * (d + 2);
    double *dout = (double *)be::dmalloc(sizeof(double) * n);
    int32_t *pos = (int32_t *)be::dmalloc(sizeof(int32_t) * P);
    int rc = 0;
    if (!dout || !pos) rc = fail(DEMCMC_ENOMEM, "chain staging does not fit on the device");
    if (!rc && (be::dzero(dout, sizeof(double) * n) ||
                be::launch_chains(h->hist_theta, h->hist_w, h->hist_acc, h->hist_id, cur_row(h).id, pos, row0, n_rows, (int32_t)P, (int32_t)d,
                                  h->cfg.group_begin * h->cfg.Np, dout) ||
                be::d2h(out, dout, sizeof(double) * n)))
        rc = fail(DEMCMC_ECUDA, "chain gather: %s", be::last_error());
    be::dfree(dout); be::dfree(pos);
    return rc;
}

int demcmc_get_history_by_slot(demcmc_handle *h, int64_t row0, int64_t n_rows, double *theta, double *w, int32_t *ids, uint8_t *acc)
{
    if (h && h->multi) {
        const size_t dd = h->d;
        if (int rc = multi_interleave(h, theta, n_rows, dd, [&](demcmc_handle *k, double *o) { return demcmc_get_history_by_slot(k, row0, n_rows, o, nullptr, nullptr, nullptr); })) return rc;
        if (int rc = multi_interleave(h, w, n_rows, 1, [&](demcmc_handle *k, double *o) { return demcmc_get_history_by_slot(k, row0, n_rows, nullptr, o, nullptr, nullptr); })) return rc;
        if (int rc = multi_interleave(h, ids, n_rows, 1, [&](demcmc_handle *k, int32_t *o) { return demcmc_get_history_by_slot(k, row0, n_rows, nullptr, nullptr, o, nullptr); })) return rc;
        return multi_interleave(h, acc, n_rows, 1, [&](demcmc_handle *k, uint8_t *o) { return demcmc_get_history_by_slot(k, row0, n_rows, nullptr, nullptr, nullptr, o); });
    }
    if (!h || row0 < 0 || n_rows < 0 || row0 + n_rows > stored_rows(h) - h->n0) return fail(DEMCMC_EINVAL, "row range outside the stored iterations");
    BE(be::set_device(h->cfg.device));
    const size_t P = h->P, d = h->d;
    if (n_rows == 0) return 0;
    row0 += h->n0;                                           // rows of the iterations come after the n_initial rows
    if (theta) BE(be::d2h(theta, h->hist_theta + row0 * P * d, sizeof(double) * n_rows * P * d));
    if (w) BE(be::d2h(w, h->hist_w + row0 * P, sizeof(double) * n_rows * P));
    if (ids) BE(be::d2h(ids, h->hist_id + row0 * P, sizeof(int32_t) * n_rows * P));
    if (acc) BE(be::d2h(acc, h->hist_acc + row0 * P, n_rows * P));
    return 0;
}

int demcmc_get_state(demcmc_handle *h, double *theta, double *weight, int32_t *ids)
{
    if (!h || !h->has_state) return fail(DEMCMC_ESTATE, "no state");
    if (h->multi)
        return for_kids(h, [&](demcmc_handle *k, int) {
            const size_t pb = (size_t)k->cfg.group_begin * k->cfg.Np;
            return demcmc_get_state(k, theta ? theta + pb * h->d : nullptr, weight ? weight + pb : nullptr, ids ? ids + pb : nullptr);
        }, false);
    BE(be::set_device(h->cfg.device));
    Row r = cur_row(h);
    const size_t P = h->P, d = h->d;
    if (theta) BE(be::d2h(theta, r.theta, sizeof(double) * P * d));
    if (weight) BE(be::d2h(weight, r.w, sizeof(double) * P));
    if (ids) BE(be::d2h(ids, r.id, sizeof(int32_t) * P));
    return 0;
}

int demcmc_get_trace(demcmc_handle *h, double *prop_theta, double *prop_weight, double *log_adj, uint8_t *accepted)
{
    if (!h) return fail(DEMCMC_EINVAL, "null handle");
    if (h->multi) {
        const int64_t S = h->kids[0]->tr_sweeps;
        if (!S) return fail(DEMCMC_ESTATE, "no trace: create the handle with cfg.trace = 1 and run first");
        if (int rc = multi_interleave(h, prop_theta, S, (size_t)h->d, [&](demcmc_handle *k, double *o) { return demcmc_get_trace(k, o, nullptr, nullptr, nullptr); })) return rc;
        if (int rc = multi_interleave(h, prop_weight, S, 1, [&](demcmc_handle *k, double *o) { return demcmc_get_trace(k, nullptr, o, nullptr, nullptr); })) return rc;
        if (int rc = multi_interleave(h, log_adj, S, 1, [&](demcmc_handle *k, double *o) { return demcmc_get_trace(k, nullptr, nullptr, o, nullptr); })) return rc;
        return multi_interleave(h, accepted, S, 1, [&](demcmc_handle *k, uint8_t *o) { return demcmc_get_trace(k, nullptr, nullptr, nullptr, o); });
    }
    if (!h->tr_sweeps) return fail(DEMCMC_ESTATE, "no trace: create the handle with cfg.trace = 1 and run first");
    BE(be::set_device(h->cfg.device));
    const size_t n = (size_t)h->tr_sweeps * h->P;
    if (prop_theta) BE(be::d2h(prop_theta, h->tr_theta, sizeof(double) * n * h->d));
    if (prop_weight) BE(be::d2h(prop_weight, h->tr_w, sizeof(double) * n));
    if (log_adj) BE(be::d2h(log_adj, h->tr_adj, sizeof(double) * n));
    if (accepted) BE(be::d2h(accepted, h->tr_acc, n));
    return 0;
}

int demcmc_get_trace_xdot(demcmc_handle *h, double *xdot)
{
    if (!h || !xdot) return fail(DEMCMC_EINVAL, "null argument");
    if (h->multi) return multi_interleave(h, xdot, h->kids[0]->tr_sweeps, 1, [&](demcmc_handle *k, double *o) { return demcmc_get_trace_xdot(k, o); });
    if (!h->tr_sweeps || !h->tr_xdot) return fail(DEMCMC_ESTATE, "no cross-term trace: MVNORMAL / HIER_NORMAL handle created with cfg.trace = 1, after a run");
    BE(be::set_device(h->cfg.device));
    BE(be::d2h(xdot, h->tr_xdot, sizeof(double) * (size_t)h->tr_sweeps * h->P));
    return 0;
}

int demcmc_set_sufficient_stat(demcmc_handle *h, int32_t on)
{
    if (!h) return fail(DEMCMC_EINVAL, "null handle");
    if (h->multi) return for_kids(h, [&](demcmc_handle *k, int) { return demcmc_set_sufficient_stat(k, on); }, false);
    if (on && h->has_model && h->dmodel.center_given) return fail(DEMCMC_EINVAL, "the model was centred on a caller-supplied vector: its cross term is not zero");
    h->suffstat = on != 0;
    return 0;
}

int demcmc_get_migration(demcmc_handle *h, int32_t *slots)
{
    if (!h || !slots) return fail(DEMCMC_EINVAL, "null argument");
    if (h->multi) {                                          // every device logged the picks of its own groups (-1 elsewhere)
        const size_t n = (size_t)h->kids[0]->mig_log_iters * h->cfg.n_groups;
        std::vector<int32_t> tmp(std::max<size_t>(1, n));
        for (size_t i = 0; i < n; ++i) slots[i] = -1;
        for (demcmc_handle *k : h->kids) {
            if (int rc = demcmc_get_migration(k, tmp.data())) return rc;
            for (size_t i = 0; i < n; ++i) slots[i] = std::max(slots[i], tmp[i]);
        }
        return 0;
    }
    memcpy(slots, h->last_mig_slots.data(), sizeof(int32_t) * (size_t)h->mig_log_iters * h->cfg.n_groups);
    return 0;
}

int demcmc_set_timing(demcmc_handle *h, int64_t l2_flush_bytes, int32_t time_loglik)
{
    if (!h || l2_flush_bytes < 0) return fail(DEMCMC_EINVAL, "bad argument");
    if (h->multi) return for_kids(h, [&](demcmc_handle *k, int) { return demcmc_set_timing(k, l2_flush_bytes, time_loglik); }, false);
    BE(be::set_device(h->cfg.device));
    be::dfree(h->flush_buf); h->flush_buf = nullptr; h->flush_bytes = 0;
    if (l2_flush_bytes > 0) {
        h->flush_buf = be::dmalloc((size_t)l2_flush_bytes);
        if (!h->flush_buf) return fail(DEMCMC_ENOMEM, "flush buffer");
        h->flush_bytes = l2_flush_bytes;
    }
    h->time_loglik = time_loglik != 0;
    return 0;
}

int demcmc_set_blocking_schedule(demcmc_handle *h, const uint8_t *on, int64_t n)
{
    if (!h || n < 0 || (n > 0 && !on)) return fail(DEMCMC_EINVAL, "bad argument");
    if (h->multi) return for_kids(h, [&](demcmc_handle *k, int) { return demcmc_set_blocking_schedule(k, on, n); }, false);
    if (h->cfg.n_blocks <= 0) return fail(DEMCMC_EINVAL, "the handle was created without parameter blocks");
    h->block_on.assign(on, on + n);
    return 0;
}

int demcmc_set_weights(demcmc_handle *h, const double *w)
{
    if (!h || !w) return fail(DEMCMC_EINVAL, "null argument");
    if (!h->has_state) return fail(DEMCMC_ESTATE, "set_state must come before set_weights");
    if (h->multi) return for_kids(h, [&](demcmc_handle *k, int) { return demcmc_set_weights(k, w + (size_t)k->cfg.group_begin * k->cfg.Np); }, false);
    BE(be::set_device(h->cfg.device));
    BE(be::h2d(cur_row(h).w, w, sizeof(double) * (size_t)h->P));
    BE(be::sync());
    return 0;
}

int demcmc_set_iteration(demcmc_handle *h, int64_t iterations_done)
{
    if (!h || iterations_done < 0) return fail(DEMCMC_EINVAL, "bad argument");
    if (h->multi) return for_kids(h, [&](demcmc_handle *k, int) { return demcmc_set_iteration(k, iterations_done); }, false);
    if (h->iters_done > 0) return fail(DEMCMC_ESTATE, "set_iteration must come before the first run of the handle");
    h->iter_offset = iterations_done;
    return 0;
}

int demcmc_set_max_chunk(demcmc_handle *h, int32_t n_sweeps)
{
    if (!h || n_sweeps < 1) return fail(DEMCMC_EINVAL, "bad argument");
    if (h->multi) return for_kids(h, [&](demcmc_handle *k, int) { return demcmc_set_max_chunk(k, n_sweeps); }, false);
    h->max_chunk = std::min<int32_t>(n_sweeps, MAX_CHUNK);
    return 0;
}

int demcmc_set_lanes(demcmc_handle *h, int32_t n_lanes)
{
    if (!h || n_lanes < 1) return fail(DEMCMC_EINVAL, "bad argument");
    if (h->multi) return for_kids(h, [&](demcmc_handle *k, int) { return demcmc_set_lanes(k, n_lanes); }, false);
    h->n_lanes = std::min<int32_t>(n_lanes, be::MAX_LANES);
    return 0;
}

int demcmc_get_counters(demcmc_handle *h, demcmc_counters *out)
{
    if (!h || !out) return fail(DEMCMC_EINVAL, "null argument");
    if (h->multi) {                                          // work summed over the devices, time = the slowest device
        demcmc_counters c = h->kids[0]->ctr;
        for (size_t i = 1; i < h->kids.size(); ++i) {
            const demcmc_counters &k = h->kids[i]->ctr;
            c.particle_updates += k.particle_updates; c.loglike_evals += k.loglike_evals; c.kernel_launches += k.kernel_launches;
            c.levels += k.levels; c.persistent_chunks += k.persistent_chunks;   // (mailbox_events / cross_migrations: the same on every device)
            c.device_ms = std::max(c.device_ms, k.device_ms); c.loglike_ms = std::max(c.loglike_ms, k.loglike_ms);
        }
        *out = c;
        return 0;
    }
    *out = h->ctr;
    return 0;
}

static int eval_impl(demcmc_handle *h, const double *theta, int64_t n, double *loglike, double *prior, double *xdot);
int demcmc_eval(demcmc_handle *h, const double *theta, int64_t n, double *loglike, double *prior) { return eval_impl(h, theta, n, loglike, prior, nullptr); }
int demcmc_eval_xdot(demcmc_handle *h, const double *theta, int64_t n, double *xdot)
{
    if (!xdot) return fail(DEMCMC_EINVAL, "null out");
    if (h && h->has_model && !is_ssd(h->dmodel.kind)) return fail(DEMCMC_EINVAL, "only MVNORMAL / HIER_NORMAL have a cross term");
    return eval_impl(h, theta, n, nullptr, nullptr, xdot);
}
static int eval_impl(demcmc_handle *h, const double *theta, int64_t n, double *loglike, double *prior, double *xdot)
{
    if (!h || !theta || n < 0) return fail(DEMCMC_EINVAL, "bad argument");
    if (!h->has_model) return fail(DEMCMC_ESTATE, "set_model first");
    if (h->multi) return eval_impl(h->kids[0], theta, n, loglike, prior, xdot);
    BE(be::set_device(h->cfg.device));
    if (n == 0) return 0;
    const size_t d = h->d, ns = (size_t)h->dmodel.n_osplit * h->dmodel.n_ksplit;
    double *dt = (double *)be::dmalloc(sizeof(double) * n * d), *dl = (double *)be::dmalloc(sizeof(double) * n),
           *dp = (double *)be::dmalloc(sizeof(double) * n), *part = (double *)be::dmalloc(sizeof(double) * n * ns),
           *dx = (double *)be::dmalloc(sizeof(double) * n);
    int rc = 0;
    if (!dt || !dl || !dp || !part || !dx) rc = fail(DEMCMC_ENOMEM, "eval staging does not fit");
    if (!rc && (be::h2d(dt, theta, sizeof(double) * n * d) || be::sync() ||
                be::launch_eval(h->dcfg, h->dmodel, dt, n, dl, dp, nullptr, part, dx) ||
                (loglike && be::d2h(loglike, dl, sizeof(double) * n)) || (prior && be::d2h(prior, dp, sizeof(double) * n)) ||
                (xdot && be::d2h(xdot, dx, sizeof(double) * n))))
        rc = fail(DEMCMC_ECUDA, "eval: %s", be::last_error());
    be::dfree(dt); be::dfree(dl); be::dfree(dp); be::dfree(part); be::dfree(dx);
    return rc;
}


int demcmc_op_project(int device, const double *p1, const double *p2, int32_t d, double *out)
{
    if (!p1 || !p2 || !out || d < 1) return fail(DEMCMC_EINVAL, "bad argument");
    if (int rc = op_begin(device)) return rc;
    DevBuf b;
    double *a = b.up(p1, d), *c = b.up(p2, d), *o = b.up<double>(nullptr, d);
    if (!a || !c || !o) return fail(DEMCMC_ENOMEM, "alloc");
    BE(be::sync());
    BE(be::launch_op_project(a, c, d, o));
    BE(be::d2h(out, o, sizeof(double) * d));
    return 0;
}

int demcmc_op_reset(int device, const double *prop, const double *pt, const uint8_t *mask, int32_t d, double *out)
{
    if (!prop || !pt || !mask || !out || d < 1) return fail(DEMCMC_EINVAL, "bad argument");
    if (int rc = op_begin(device)) return rc;
    DevBuf b;
    double *a = b.up(prop, d), *c = b.up(pt, d), *o = b.up<double>(nullptr, d);
    uint8_t *m = b.up(mask, d);
    if (!a || !c || !o || !m) return fail(DEMCMC_ENOMEM, "alloc");
    BE(be::sync());
    BE(be::launch_op_reset(a, c, m, d, o));
    BE(be::d2h(out, o, sizeof(double) * d));
    return 0;
}

int demcmc_op_de_proposal(int device, const double *pt, const double *pm, const double *pn, const double *pb,
                          double g1, double g2, const double *bn, int32_t d, double *out)
{
    if (!pt || !pm || !pn || !bn || !out || d < 1) return fail(DEMCMC_EINVAL, "bad argument");
    if (int rc = op_begin(device)) return rc;
    DevBuf b;
    double *t = b.up(pt, d), *m = b.up(pm, d), *n = b.up(pn, d), *bb = pb ? b.up(pb, d) : nullptr, *nz = b.up(bn, d), *o = b.up<double>(nullptr, d);
    if (!t || !m || !n || !nz || !o || (pb && !bb)) return fail(DEMCMC_ENOMEM, "alloc");
    BE(be::sync());
    BE(be::launch_op_de(t, m, n, bb, g1, g2, nz, d, o));
    BE(be::d2h(out, o, sizeof(double) * d));
    return 0;
}

int demcmc_op_snooker(int device, const double *pt, const double *pz, const double *pm, const double *pn,
                      double g, const double *bn, int32_t d, double *out, double *log_adj)
{
    if (!pt || !pz || !pm || !pn || !bn || !out || d < 1) return fail(DEMCMC_EINVAL, "bad argument");
    if (int rc = op_begin(device)) return rc;
    DevBuf b;
    double *t = b.up(pt, d), *z = b.up(pz, d), *m = b.up(pm, d), *n = b.up(pn, d), *nz = b.up(bn, d), *o = b.up<double>(nullptr, d), *la = b.up<double>(nullptr, 1);
    if (!t || !z || !m || !n || !nz || !o || !la) return fail(DEMCMC_ENOMEM, "alloc");
    BE(be::sync());
    BE(be::launch_op_snooker(t, z, m, n, g, nz, d, o, la));
    BE(be::d2h(out, o, sizeof(double) * d));
    if (log_adj) BE(be::d2h(log_adj, la, sizeof(double)));
    return 0;
}

int demcmc_op_accept(int device, const double *w_prop, const double *w_cur, const double *log_adj, const double *u, int32_t n, uint8_t *out)
{
    if (!w_prop || !w_cur || !log_adj || !u || !out || n < 1) return fail(DEMCMC_EINVAL, "bad argument");
    if (int rc = op_begin(device)) return rc;
    DevBuf b;
    double *a = b.up(w_prop, n), *c = b.up(w_cur, n), *l = b.up(log_adj, n), *uu = b.up(u, n);
    uint8_t *o = b.up<uint8_t>(nullptr, n);
    if (!a || !c || !l || !uu || !o) return fail(DEMCMC_ENOMEM, "alloc");
    BE(be::sync());
    BE(be::launch_op_accept(a, c, l, uu, n, o));
    BE(be::d2h(out, o, n));
    return 0;
}

int demcmc_op_select(int device, const double *w, int32_t n, double u, int32_t *base_idx, int32_t *migrate_idx)
{
    if (!w || n < 1) return fail(DEMCMC_EINVAL, "bad argument");
    if (int rc = op_begin(device)) return rc;
    DevBuf b;
    double *a = b.up(w, n);
    int32_t *o = b.up<int32_t>(nullptr, 2);
    if (!a || !o) return fail(DEMCMC_ENOMEM, "alloc");
    BE(be::sync());
    BE(be::launch_op_select(a, n, u, o, o + 1));
    int32_t r[2];
    BE(be::d2h(r, o, sizeof r));
    if (base_idx) *base_idx = r[0];
    if (migrate_idx) *migrate_idx = r[1];
    return 0;
}

int demcmc_comm_unique_id(uint8_t id[128])
{
    if (!id) return fail(DEMCMC_EINVAL, "null id");
    if (be::comm_unique_id(id)) return fail(DEMCMC_ECOMM, "%s", be::last_error());
    return 0;
}

int demcmc_comm_init(demcmc_handle *h, const uint8_t id[128], int32_t rank, int32_t n_ranks)
{
    if (!h || !id || n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail(DEMCMC_EINVAL, "bad argument");
    if (h->multi || h->parent) return fail(DEMCMC_EINVAL, "a multi-device handle shards over the GPUs of this process by itself: demcmc_comm_init is for one handle per process");
    if (n_ranks > MAX_RANKS) return fail(DEMCMC_EUNSUPPORTED, "more than %d ranks", (int)MAX_RANKS);
    const int Gt = h->cfg.n_groups;
    if (Gt % n_ranks) return fail(DEMCMC_EINVAL, "n_groups %d is not a multiple of the %d ranks", Gt, n_ranks);
    const int per = Gt / n_ranks;
    if (h->cfg.group_begin != rank * per || h->G_local != per) return fail(DEMCMC_EINVAL, "handle holds groups [%d,%d) but rank %d of %d must hold [%d,%d)", h->cfg.group_begin, h->cfg.group_begin + h->G_local, rank, n_ranks, rank * per, rank * per + per);
    BE(be::set_device(h->cfg.device));
    if (n_ranks > 1 && be::comm_init(id, rank, n_ranks, &h->comm)) return fail(DEMCMC_ECOMM, "%s", be::last_error());
    h->rank = rank; h->n_ranks = n_ranks;
    for (int g = 0; g < Gt; ++g) h->group_owner[g] = g / per;
    // P2P migration: every rank maps every other rank's mailbox (CUDA IPC over NVLink); the handles travel through the
    // communicator.  All ranks take the same decision (two all-gathers of status bytes); any failure anywhere leaves
    // the NCCL send/recv exchange in place.
    if (n_ranks > 1 && mbox_wanted() && !h->mbox_on) {
        MboxShared &sh = g_mbox_shared[h->cfg.device];
        int depth, max_rows, row_len;
        mbox_geometry(h, &depth, &max_rows, &row_len);
        const size_t need_d = (size_t)depth * max_rows * row_len, need_f = (size_t)depth * max_rows;
        constexpr size_t REC = 136;                          // 128-byte handle blob + status byte, 8-byte aligned
        std::vector<uint8_t> mine(REC, 0), all(REC * n_ranks, 0);
        uint8_t *dsend = (uint8_t *)be::dmalloc(REC), *drecv = (uint8_t *)be::dmalloc(REC * n_ranks);
        // every rank calls gather() the same number of times whatever happened locally: the status bytes carry failures
        auto gather = [&](uint8_t status) {
            mine[128] = status;
            const bool sent = dsend && drecv && !be::h2d(dsend, mine.data(), REC) && !be::comm_allgather(h->comm, dsend, drecv, REC) &&
                              !be::d2h(all.data(), drecv, REC * n_ranks);
            int lo = 255;
            for (int r = 0; r < n_ranks; ++r) lo = std::min<int>(lo, all[REC * r + 128]);
            return sent ? lo : 0;                            // the smallest status anybody reported
        };
        const bool fits = sh.box.rows && sh.n_ranks == n_ranks && sh.rank == rank && sh.cap_doubles >= need_d && sh.cap_flags >= need_f;
        bool use = false;
        if (gather(fits ? 2 : 1) == 2) use = true;           // round 1: does everybody's cached mailbox fit this job?
        else {
            Mbox fresh = { nullptr, nullptr, 0, 0, 0 };
            const bool made = be::mbox_create(depth, max_rows, row_len, &fresh) == 0 && be::mbox_export(fresh, mine.data()) == 0;
            const bool all_made = gather(made ? 1 : 0) == 1; // round 2: everybody publishes a new mailbox
            PeerTable pt = {};
            bool opened = all_made;
            for (int r = 0; r < n_ranks && opened; ++r) {
                if (r == rank) { pt.rows[r] = fresh.rows; pt.flags[r] = fresh.flags; continue; }
                Mbox pm = { nullptr, nullptr, 0, 0, 0 };
                if (be::mbox_open(all.data() + REC * r, &pm)) opened = false;
                else { pt.rows[r] = pm.rows; pt.flags[r] = pm.flags; }
            }
            if (gather(opened ? 1 : 0) == 1) {               // round 3: everybody mapped everybody
                // (an older mailbox stays mapped by the peers: it is abandoned, never freed under them)
                sh.box = fresh; sh.peers = pt; sh.cap_doubles = need_d; sh.cap_flags = need_f; sh.n_ranks = n_ranks; sh.rank = rank;
                use = true;
            }
        }
        be::dfree(dsend); be::dfree(drecv);
        if (use) {
            h->mbox = sh.box; h->mbox.depth = depth; h->mbox.max_rows = max_rows; h->mbox.row_len = row_len;
            h->peers = sh.peers;
            h->mbox_shared = true;                            // owned by the process, not by the handle
            h->mbox_seq_p = &sh.seq;                          // ... and so is the event counter: it only ever grows
            h->mbox_on = true;
            void *comm = h->comm;
            h->mbox_barrier = [comm]() { return be::comm_barrier(comm); };
        }
    }
    return 0;
}

int demcmc_fp64_peak(int device, double *tflops)
{
    if (!tflops) return fail(DEMCMC_EINVAL, "null out");
    if (int rc = op_begin(device)) return rc;
    BE(be::fp64_peak(tflops));
    return 0;
}

int demcmc_fp64_peaks(int device, double *dfma_tflops, double *dmma_tflops)
{
    if (!dfma_tflops && !dmma_tflops) return fail(DEMCMC_EINVAL, "null out");
    if (int rc = op_begin(device)) return rc;
    BE(be::fp64_peaks(dfma_tflops, dmma_tflops));
    return 0;
}

int demcmc_copy_peak(int device, double *gbs)
{
    if (!gbs) return fail(DEMCMC_EINVAL, "null out");
    if (int rc = op_begin(device)) return rc;
    BE(be::copy_peak(gbs));
    return 0;
}

} // extern "C"

// kernels.cu -- CUDA (sm_100a) implementation of backend.h: every kernel of libdemcmc_b200.
//
//   k_propose      one warp per particle: DE / snooker / mutation proposal, kappa and block masks,
//                  bounds, prior, snooker adjustment                       (HBM-bound, ~5 d-vectors)
//   k_xdot         cross term sum_i sum_k x'_ik m'_pk of the expanded sum of squares for a tile of
//                  particles against a range of observation tiles, on the fp64 tensor path
//                  (DMMA m8n8k4): the likelihood of the isotropic MVN and the hierarchical
//                  normal models                                           (fp64-pipe-bound)
//   k_ll_pointwise per-observation log densities (Gaussian, LNR, LBA) for a tile of particles
//   k_ll_custom    the same for a density the caller writes (DEMCMC_CUSTOM), compiled at run time with NVRTC
//   k_accept       one warp per particle: fixed-order reduction of the partial sums, Metropolis
//                  accept, state-row write (replaces store_samples!)       (HBM-bound)
//   k_mig_*        migration picks and the cyclic shift
//   k_history      by-slot rows -> the reference's samples[n_rows, d, P] layout
#include <cuda_runtime.h>
#include <stddef.h>
#include <dlfcn.h>
#include <nvrtc.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "backend.h"
#include "de_particle.h"

namespace de {
namespace be {

// Threading: one host thread drives one device at a time (a multi-device handle runs one thread per device,
// engine.cpp).  What is "current" (device, lane, launch counter) is thread-local; what belongs to a device
// (streams, events, staging buffers, the NCCL communicator) lives in per-device slots whose lazy creation is
// serialised by g_mu.  Two handles on the SAME device must not be driven from two threads at once.
static std::mutex g_mu;
static thread_local std::string g_be_err;
static thread_local int64_t g_launches = 0;
static thread_local int g_dev = 0;
// Lanes: independent sets of groups run as concurrent kernel chains, one stream per lane, so the
// likelihood kernel of one lane covers the propose / accept latency of the other (engine.cpp).
// Lane 0 is the engine stream; every copy, event and one-off kernel runs there.
static thread_local int g_lane = 0;
static cudaStream_t g_stream[64][MAX_LANES] = { { nullptr } };
static cudaEvent_t g_lane_ev[64][MAX_LANES] = { { nullptr } };
static cudaEvent_t g_t0[64] = { nullptr }, g_t1[64] = { nullptr };

static int cu_fail(cudaError_t e, const char *what)
{
    g_be_err = std::string(what) + ": " + cudaGetErrorString(e);
    return -1;
}
#define CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return cu_fail(e_, #call); } while (0)
#define LAUNCHED(name) do { ++g_launches; cudaError_t e_ = cudaGetLastError(); if (e_ != cudaSuccess) return cu_fail(e_, name); } while (0)

static cudaStream_t stream()
{
    if (!g_stream[g_dev][g_lane]) {
        std::lock_guard<std::mutex> lk(g_mu);
        if (!g_stream[g_dev][g_lane]) cudaStreamCreateWithFlags(&g_stream[g_dev][g_lane], cudaStreamNonBlocking);
    }
    return g_stream[g_dev][g_lane];
}

// Kernels of one level are chained with programmatic dependent launch: the next kernel's CTAs may
// become resident and run their state-independent prologue while the previous kernel drains; each
// kernel executes griddepcontrol.wait before it touches anything an earlier kernel wrote.
// DEMCMC_NO_PDL=1 falls back to plain stream order (A/B measurements).
static bool use_pdl()
{
    static int v = -1;
    if (v < 0) { const char *e = getenv("DEMCMC_NO_PDL"); v = (e && e[0] == '1') ? 0 : 1; }
    return v == 1;
}
// set by launch_plan: the next kernel on lane 0 reads the plan records BEFORE its griddepcontrol.wait, so it must not be
// chained to k_plan programmatically (the other lanes start behind an event recorded after k_plan)
static thread_local bool g_break_chain = false;
template <typename... KArgs, typename... Args>
static cudaError_t launch_chained(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream();
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = (use_pdl() && !(g_break_chain && g_lane == 0)) ? 1 : 0;
    if (g_lane == 0) g_break_chain = false;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// ---- debug timeline (DEMCMC_TIMELINE=<levels> DEMCMC_TIMELINE_FILE=<csv>): every kernel of a level
// stamps %globaltimer into one 16-word slot, so the gaps between the kernels of a PDL chain can be
// read without events (which would break the chain) and without a profiler (which serialises it)
enum { TL_P0 = 0, TL_P1, TL_X0, TL_X0MAX, TL_XWAIT, TL_XFIRST, TL_XLOOP0, TL_XLOOP1, TL_X1, TL_A0, TL_A1, TL_N, TL_PW, TL_AW, TL_Q0, TL_Q1, TL_Q2, TL_Q3, TL_WORDS = 24 };
static unsigned long long *g_tl = nullptr;
static int g_tl_cap = -1, g_tl_level = 0, g_tl_cta_level = -1;
constexpr int TL_CTA_WORDS = 4, TL_CTA_MAX = 4096;
static unsigned long long *tl_cta()      // per-CTA stamps of the one level named by DEMCMC_TIMELINE_CTA
{
    return (g_tl_cap > 0 && g_tl && g_tl_level == g_tl_cta_level) ? g_tl + (size_t)TL_WORDS * g_tl_cap : nullptr;
}
static unsigned long long *tl_slot()
{
    if (g_tl_cap < 0) {
        const char *e = getenv("DEMCMC_TIMELINE");
        g_tl_cap = e ? atoi(e) : 0;
        const size_t words = (size_t)TL_WORDS * g_tl_cap + (size_t)TL_CTA_WORDS * TL_CTA_MAX;
        if (g_tl_cap > 0 && (cudaMalloc(&g_tl, sizeof(unsigned long long) * words) != cudaSuccess ||
                             cudaMemset(g_tl, 0, sizeof(unsigned long long) * words) != cudaSuccess)) g_tl_cap = 0;
        if (const char *c = getenv("DEMCMC_TIMELINE_CTA")) g_tl_cta_level = atoi(c);
    }
    return (g_tl_cap > 0 && g_tl_level < g_tl_cap) ? g_tl + (size_t)TL_WORDS * g_tl_level : nullptr;
}
static void pk_timeline_dump();
void timeline_dump()
{
    pk_timeline_dump();
    if (g_tl_cap <= 0 || !g_tl) return;
    const char *path = getenv("DEMCMC_TIMELINE_FILE");
    if (!path) return;
    cudaDeviceSynchronize();
    const int n = g_tl_level < g_tl_cap ? g_tl_level : g_tl_cap;
    std::vector<unsigned long long> h((size_t)TL_WORDS * (n > 0 ? n : 1));
    if (n <= 0 || cudaMemcpy(h.data(), g_tl, sizeof(unsigned long long) * TL_WORDS * n, cudaMemcpyDeviceToHost) != cudaSuccess) return;
    FILE *f = fopen(path, "w");
    if (!f) return;
    fprintf(f, "level,n,propose_start,propose_end,xdot_start,xdot_last_start,xdot_wait_done,xdot_first_data,xdot_loop_end_min,xdot_loop_end_max,xdot_end,accept_start,accept_end,propose_wait_done,accept_wait_done,q0,q1,q2,q3\n");
    const unsigned long long t0 = ~h[TL_P0];
    for (int i = 0; i < n; ++i) {
        const unsigned long long *w = h.data() + (size_t)TL_WORDS * i;
        auto rel = [&](unsigned long long v) { return (double)((long long)(v - t0)) * 1e-3; };
        fprintf(f, "%d,%llu,%.3f,%.3f,%.3f,%.3f,%.3f,%.3f,%.3f,%.3f,%.3f,%.3f,%.3f,%.3f,%.3f,%.3f,%.3f,%.3f,%.3f\n", i, w[TL_N], rel(~w[TL_P0]), rel(w[TL_P1]), rel(~w[TL_X0]), rel(w[TL_X0MAX]),
                rel(w[TL_XWAIT]), rel(w[TL_XFIRST]), rel(~w[TL_XLOOP0]), rel(w[TL_XLOOP1]), rel(w[TL_X1]), rel(~w[TL_A0]), rel(w[TL_A1]), rel(~w[TL_PW]), rel(~w[TL_AW]), rel(w[TL_Q0]), rel(w[TL_Q1]), rel(w[TL_Q2]), rel(w[TL_Q3]));
    }
    fclose(f);
    if (g_tl_cta_level >= 0) {
        std::vector<unsigned long long> c((size_t)TL_CTA_WORDS * TL_CTA_MAX);
        if (cudaMemcpy(c.data(), g_tl + (size_t)TL_WORDS * g_tl_cap, sizeof(unsigned long long) * c.size(), cudaMemcpyDeviceToHost) == cudaSuccess) {
            std::string p2 = std::string(path) + ".cta";
            FILE *g = fopen(p2.c_str(), "w");
            if (g) {
                fprintf(g, "cta,start,wait_done,loop_end,tiles\n");
                unsigned long long c0 = ~0ull;
                for (int i = 0; i < TL_CTA_MAX; ++i) if (c[(size_t)i * 4]) c0 = c[(size_t)i * 4] < c0 ? c[(size_t)i * 4] : c0;
                for (int i = 0; i < TL_CTA_MAX; ++i) if (c[(size_t)i * 4])
                    fprintf(g, "%d,%.3f,%.3f,%.3f,%llu\n", i, (double)(c[(size_t)i * 4] - c0) * 1e-3, (double)(c[(size_t)i * 4 + 1] - c0) * 1e-3, (double)(c[(size_t)i * 4 + 2] - c0) * 1e-3, c[(size_t)i * 4 + 3]);
                fclose(g);
            }
        }
    }
}
__device__ __forceinline__ unsigned long long gtime()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void tl_min(unsigned long long *tl, int w) { if (tl) atomicMax(tl + w, ~gtime()); }
__device__ __forceinline__ void tl_max(unsigned long long *tl, int w) { if (tl) atomicMax(tl + w, gtime()); }

void set_lane(int lane) { g_lane = (lane >= 0 && lane < MAX_LANES) ? lane : 0; }
static cudaEvent_t lane_event(int lane)
{
    if (!g_lane_ev[g_dev][lane]) cudaEventCreateWithFlags(&g_lane_ev[g_dev][lane], cudaEventDisableTiming);
    return g_lane_ev[g_dev][lane];
}
int lane_fork(int n_lanes)
{
    if (n_lanes < 2) return 0;
    const int keep = g_lane;
    g_lane = 0;
    cudaStream_t s0 = stream();
    CU(cudaEventRecord(lane_event(0), s0));
    for (int l = 1; l < n_lanes && l < MAX_LANES; ++l) { g_lane = l; CU(cudaStreamWaitEvent(stream(), lane_event(0), 0)); }
    g_lane = keep;
    return 0;
}
int lane_join(int n_lanes)
{
    if (n_lanes < 2) return 0;
    const int keep = g_lane;
    g_lane = 0;
    cudaStream_t s0 = stream();
    for (int l = 1; l < n_lanes && l < MAX_LANES; ++l) {
        g_lane = l;
        CU(cudaEventRecord(lane_event(l), stream()));
        CU(cudaStreamWaitEvent(s0, lane_event(l), 0));
    }
    g_lane = keep;
    return 0;
}

const char *name() { return "cuda-sm100a"; }
const char *last_error() { return g_be_err.c_str(); }
int device_count()
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { cu_fail(e, "cudaGetDeviceCount"); return 0; }
    return n;
}
int set_device(int dev)
{
    if (dev < 0 || dev >= 64) { g_be_err = "device ordinal out of range"; return -1; }
    CU(cudaSetDevice(dev));
    g_dev = dev;
    return 0;
}
// Device memory comes from the stream-ordered allocator with an unbounded release threshold: a
// handle that is destroyed leaves its blocks in the pool, so creating the next one (one handle per
// sample() call) costs microseconds instead of a cudaMalloc / cudaFree pair per buffer.
static void pool_setup()
{
    static bool done[64] = { false };
    if (done[g_dev]) return;
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, g_dev) == cudaSuccess) {
        unsigned long long keep = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    done[g_dev] = true;
}
void *dmalloc(size_t bytes)
{
    pool_setup();
    void *p = nullptr;
    cudaError_t e = cudaMallocAsync(&p, bytes ? bytes : 8, stream());
    if (e != cudaSuccess) { cu_fail(e, "cudaMallocAsync"); return nullptr; }
    return p;
}
void dfree(void *p) { if (p) cudaFreeAsync(p, stream()); }
// outside the pool: cudaDeviceEnablePeerAccess covers it directly (a 662 MB pool allocation that seven peers must map
// failed with "out of memory" on an 8-GPU box)
void *dmalloc_shared(size_t bytes)
{
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes ? bytes : 8);
    if (e != cudaSuccess) { cu_fail(e, "cudaMalloc"); return nullptr; }
    return p;
}
void dfree_shared(void *p) { if (p) { cudaStreamSynchronize(stream()); cudaFree(p); } }
// pinned blocks are recycled through a small free list for the same reason
struct PinnedBlock { void *p; size_t bytes; bool busy; };
static std::vector<PinnedBlock> g_pinned;
void *hmalloc_pinned(size_t bytes)
{
    if (!bytes) bytes = 8;
    std::lock_guard<std::mutex> lk(g_mu);
    for (auto &b : g_pinned)
        if (!b.busy && b.bytes >= bytes && b.bytes <= 2 * bytes + 4096) { b.busy = true; return b.p; }
    void *p = nullptr;
    cudaError_t e = cudaMallocHost(&p, bytes);
    if (e != cudaSuccess) { cu_fail(e, "cudaMallocHost"); return nullptr; }
    g_pinned.push_back({ p, bytes, true });
    return p;
}
void hfree_pinned(void *p)
{
    if (!p) return;
    std::lock_guard<std::mutex> lk(g_mu);
    for (auto &b : g_pinned) if (b.p == p) { b.busy = false; return; }
    cudaFreeHost(p);
}
// (Uploads stay on the driver's pageable path: 40 MB of numpy memory arrive in 2-3 ms either way -- a pipelined pinned staging
// like d2h_staged below was measured and made no difference.)
int h2d(void *dst, const void *src, size_t bytes) { if (bytes) CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream())); return 0; }
// Large downloads (the chains of a run: hundreds of MB into a freshly allocated, never-touched
// caller buffer) do not go through the driver's pageable path -- measured on the B200 box it takes
// anything from 57 ms to 2.2 s for the same 217 MB, depending on how the destination pages fault.
// They are pipelined through two pinned staging blocks instead: chunk c+1 crosses PCIe while four
// host threads copy chunk c into the caller's pages (the first touch of those pages is the cost).
static int d2h_staged(void *dst, const void *src, size_t bytes)
{
    constexpr size_t CHUNK = (size_t)16 << 20;
    constexpr int NT = 4;
    static void *stage[64][2] = { { nullptr } };
    static cudaEvent_t done[64][2] = { { nullptr } };
    for (int b = 0; b < 2; ++b) {
        if (!stage[g_dev][b]) CU(cudaMallocHost(&stage[g_dev][b], CHUNK));
        if (!done[g_dev][b]) CU(cudaEventCreateWithFlags(&done[g_dev][b], cudaEventDisableTiming));
    }
    const size_t n_chunks = (bytes + CHUNK - 1) / CHUNK;
    auto issue = [&](size_t c) -> cudaError_t {
        const size_t off = c * CHUNK, len = std::min(CHUNK, bytes - off);
        cudaError_t e = cudaMemcpyAsync(stage[g_dev][c & 1], (const char *)src + off, len, cudaMemcpyDeviceToHost, stream());
        return e != cudaSuccess ? e : cudaEventRecord(done[g_dev][c & 1], stream());
    };
    CU(issue(0));
    for (size_t c = 0; c < n_chunks; ++c) {
        CU(cudaEventSynchronize(done[g_dev][c & 1]));
        if (c + 1 < n_chunks) CU(issue(c + 1));                  // the other block: its host copy finished last round
        const size_t off = c * CHUNK, len = std::min(CHUNK, bytes - off);
        const char *from = (const char *)stage[g_dev][c & 1];
        char *to = (char *)dst + off;
        std::thread th[NT];
        const size_t part = ((len / NT) + 4095) & ~(size_t)4095;
        for (int t = 0; t < NT; ++t) {
            const size_t o = std::min(len, (size_t)t * part), l = std::min(part, len - o);
            th[t] = std::thread([=]() { if (l) memcpy(to + o, from + o, l); });
        }
        for (int t = 0; t < NT; ++t) th[t].join();
    }
    return 0;
}
int d2h(void *dst, const void *src, size_t bytes)
{
    if (!bytes) return 0;
    static long long staged_min = -1;
    if (staged_min < 0) { const char *e = getenv("DEMCMC_D2H_STAGED_MIN_MB"); staged_min = (long long)(e ? atoi(e) : 4) << 20; }   // 8.7 MB of chains: 3.3 ms through the driver's pageable path, 1.2-1.8 ms staged
    if ((long long)bytes >= staged_min) {
        // a page-locked destination (Handle.chains() allocates one when it can) takes the copy engine directly
        cudaPointerAttributes at;
        const bool pinned = cudaPointerGetAttributes(&at, dst) == cudaSuccess && at.type == cudaMemoryTypeHost;
        if (!pinned) { (void)cudaGetLastError(); return d2h_staged(dst, src, bytes); }
    }
    CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, stream()));
    CU(cudaStreamSynchronize(stream()));
    return 0;
}
int d2d(void *dst, const void *src, size_t bytes) { if (bytes) CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, stream())); return 0; }
int dzero(void *dst, size_t bytes) { if (bytes) CU(cudaMemsetAsync(dst, 0, bytes, stream())); return 0; }
int sync() { CU(cudaStreamSynchronize(stream())); return 0; }
void *event_create()
{
    cudaEvent_t e = nullptr;
    if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    return (void *)e;
}
void event_destroy(void *ev) { if (ev) cudaEventDestroy((cudaEvent_t)ev); }
int event_record(void *ev) { CU(cudaEventRecord((cudaEvent_t)ev, stream())); return 0; }
int event_wait(void *ev) { CU(cudaEventSynchronize((cudaEvent_t)ev)); return 0; }
void *tevent_create()
{
    cudaEvent_t e = nullptr;
    if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
    return (void *)e;
}
void tevent_destroy(void *ev) { if (ev) cudaEventDestroy((cudaEvent_t)ev); }
int tevent_elapsed(void *a, void *b, double *ms)
{
    float f = 0.f;
    CU(cudaEventElapsedTime(&f, (cudaEvent_t)a, (cudaEvent_t)b));
    *ms = f;
    return 0;
}
int dfill(void *dst, int byte, size_t bytes) { if (bytes) CU(cudaMemsetAsync(dst, byte, bytes, stream())); return 0; }
int timer_start()
{
    if (!g_t0[g_dev]) { CU(cudaEventCreate(&g_t0[g_dev])); CU(cudaEventCreate(&g_t1[g_dev])); }
    CU(cudaEventRecord(g_t0[g_dev], stream()));
    return 0;
}
int timer_stop(double *ms)
{
    CU(cudaEventRecord(g_t1[g_dev], stream()));
    CU(cudaEventSynchronize(g_t1[g_dev]));
    float f = 0.f;
    CU(cudaEventElapsedTime(&f, g_t0[g_dev], g_t1[g_dev]));
    *ms = f;
    return 0;
}
int64_t launch_count() { return g_launches; }

// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

struct WarpLanes {
    __device__ __forceinline__ int lane() const { return threadIdx.x & 31; }
    __device__ __forceinline__ int width() const { return 32; }
    __device__ __forceinline__ double sum(double x) const { return warp_sum(x); }
    __device__ __forceinline__ bool all(bool b) const { return __all_sync(0xffffffffu, b) != 0; }
    __device__ __forceinline__ int min_int(int x) const { return __reduce_min_sync(0xffffffffu, x); }
    __device__ __forceinline__ void sync() const { __syncwarp(); }
    // programmatic dependent launch: everything before this point touches only data that is constant
    // for the whole chunk (schedule, tape, Philox); the state written by earlier kernels comes after
    __device__ __forceinline__ void dependency_wait() const { asm volatile("griddepcontrol.wait;\n" ::: "memory"); }
};
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;\n" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory"); }

struct ksum_t { double s, c; };
__device__ __forceinline__ void kadd(ksum_t &k, double x)
{
    const double t = k.s + x;
    if (isfinite(t)) { if (fabs(k.s) >= fabs(x)) k.c += (k.s - t) + x; else k.c += (x - t) + k.s; }
    k.s = t;
}
__device__ __forceinline__ double kval(const ksum_t &k) { return isfinite(k.s) ? k.s + k.c : k.s; }

// ------------------------------------------------------------------------------------------------
// propose / accept: one warp per particle of the level
// ------------------------------------------------------------------------------------------------
constexpr int PA_THREADS = 128;

// per-device staging for k_xdot: the proposals' centred means as DMMA B fragments,
// bfrag[octet of the level][dimension split][k-step j][lane], and the fixed-point magic constant of
// every particle of the level, magic[level order]
struct XdStage { double *bfrag = nullptr; double *magic = nullptr; size_t cap = 0; bool fresh = false; long long geom = -1; };   // fresh: cleared on its lane's stream just now
static XdStage g_xs[64][MAX_LANES];
static XdStage *xd_stage(const ModelDev &m, int n);

// leaves one parameter vector's centred means where k_xdot wants them, together with the particle's
// fixed-point scale (de_math.h: xd_scale); wi = rank of the particle in the launch
__device__ __forceinline__ void stage_scale(const ModelDev &m, double msq, int64_t wi, double *magic, long long *acc, double *q, double *msq_out)
{
    if ((threadIdx.x & 31) == 0) {
        const XdScale sc = xd_scale(msq, m.ssd_rowmax, m.ssd_qbits);
        magic[wi] = sc.magic;
        *q = sc.q;
        *acc = 0;
        if (msq_out) *msq_out = msq;
    }
}
// where dimension k of the wi-th particle of a launch goes: base (per particle) + offset (per dimension), the latter in
// 32-bit arithmetic with the division by the split length done by multiplication (ModelDev::ksplit_magic) -- the plain
// 64-bit form with a hardware-less integer division cost 57 instructions per element, a tenth of the wide proposal kernel
__device__ __forceinline__ size_t bfrag_base(const ModelDev &m, int64_t wi)
{
    return (size_t)(wi / SSD_OCT) * (size_t)(m.n_ksplit * m.ssd_nj * 32);
}
__device__ __forceinline__ uint32_t bfrag_offset(const ModelDev &m, int n, int k)
{
    const int ks = m.n_ksplit == 1 ? 0 : (int)__umulhi((uint32_t)k, m.ksplit_magic), kl = k - ks * m.ksplit_len;
    const uint32_t frag = (uint32_t)(ks * m.ssd_nj + (kl >> 2)) * 32u;
    if (m.debug_corrupt) {                                   // mutation tests only (de_types.h: debug_corrupt)
        if (m.debug_corrupt == 1) return frag + (kl & 3) * 8 + n;
        if (m.debug_corrupt == 3 && m.ssd_nj > 1 && (kl >> 2) == m.ssd_nj - 1) return frag - 32 + n * 4 + (kl & 3);
    }
    return frag + n * 4 + (kl & 3);
}
__device__ __forceinline__ size_t bfrag_index(const ModelDev &m, int64_t wi, int k)
{
    return bfrag_base(m, wi) + bfrag_offset(m, (int)(wi % SSD_OCT), k);
}
__device__ __forceinline__ void stage_bfrag(const ModelDev &m, const double *theta, int64_t wi, double *bfrag, double *magic,
                                            long long *acc, double *q, double *msq_out)
{
    const int lane = threadIdx.x & 31;
    double msq = 0.0;
    for (int k = lane; k < m.ssd_k; k += 32) {
        const double v = centred_mean(m, theta, k);
        msq += v * v;
        bfrag[bfrag_index(m, wi, k)] = v;
    }
    stage_scale(m, warp_sum(msq), wi, magic, acc, q, msq_out);
}

// the MVN model's means ARE proposal elements: stage them while they are still in registers
// (the data centre of the lane's first elements is fetched before the dependency wait)
struct StageSink {
    const ModelDev &m;
    double *bfrag;
    int64_t wi;
    bool on;
    double cen[PROP_PRE];
    double msq;
    __device__ __forceinline__ void prefetch(int q, int k) { if (on && k < m.ssd_k) cen[q] = m.center[k]; }
    __device__ __forceinline__ void elem(int q, int k, double v)
    {
        if (!on || k >= m.ssd_k) return;
        const double c = v - (q < PROP_PRE ? cen[q] : m.center[k]);
        msq += c * c;
        bfrag[bfrag_index(m, wi, k)] = c;
    }
};

__global__ void __launch_bounds__(PA_THREADS) k_propose(ConfigDev cfg, ModelDev m, Level lv, double *bfrag, double *magic, unsigned long long *tl)
{
    pdl_launch_dependents();
    if ((threadIdx.x & 31) == 0) tl_min(tl, TL_P0);
    const int wi = (blockIdx.x * PA_THREADS + threadIdx.x) >> 5;
    if (wi >= lv.n) { pdl_wait(); return; }
    const uint32_t e = (uint32_t)lv.order[wi];
    const SweepCtx ctx = lv.ctxs[e >> LV_SLOT_SHIFT];
    const int p = (int)(e & LV_POS_MASK);
    StageSink sink = { m, bfrag, wi, bfrag != nullptr && m.kind == M_MVNORMAL, { 0.0 }, 0.0 };
    propose_particle(WarpLanes(), cfg, m, ctx, p, sink);
    if (bfrag) {
        if (sink.on) stage_scale(m, warp_sum(sink.msq), wi, magic, ctx.ll_acc + p, ctx.ll_q + p, ctx.prop_msq + p);
        else {
            __syncwarp();
            stage_bfrag(m, ctx.prop_theta + (size_t)p * cfg.d, wi, bfrag, magic, ctx.ll_acc + p, ctx.ll_q + p, ctx.prop_msq + p);
        }
    }
    if ((threadIdx.x & 31) == 0) { tl_max(tl, TL_P1); if (tl && wi == 0) tl[TL_N] = (unsigned long long)lv.n; }
}

// TEMPER: the power-posterior terms (a tempered handle); untempered handles launch k_accept<false>, which keeps its registers
template <bool TEMPER>
__global__ void __launch_bounds__(PA_THREADS) k_accept(ConfigDev cfg, ModelDev m, Level lv, unsigned long long *tl)
{
    pdl_launch_dependents();
    if ((threadIdx.x & 31) == 0) tl_min(tl, TL_A0);
    const int wi = (blockIdx.x * PA_THREADS + threadIdx.x) >> 5;
    if (wi >= lv.n) { pdl_wait(); return; }
    const uint32_t e = (uint32_t)lv.order[wi];
    const SweepCtx ctx = lv.ctxs[e >> LV_SLOT_SHIFT];
    accept_particle<WarpLanes, TEMPER>(WarpLanes(), cfg, m, ctx, (int)(e & LV_POS_MASK));
    if ((threadIdx.x & 31) == 0) tl_max(tl, TL_A1);
}

// ---- wide variants: one CTA of PAW_THREADS threads per particle when the parameter vector is long
// (hierarchical normal with 1000 subjects: d = 1003).  With one warp per particle the proposal is a
// 32-iteration chain of dependent loads, Philox draws and prior terms per lane (90 us per level on
// configs[3]); eight warps cut the chain to four iterations.  Same per-element arithmetic
// (de_particle.h), block-wide reductions in a fixed order.
constexpr int PAW_MIN_D = 256;           // parameter count from which the wide kernels are used

template <int PAW_THREADS>
struct BlockLanes {
    double *red;                          // shared scratch: PAW_THREADS / 32 doubles
    int *ired;
    unsigned long long *tl;               // debug timeline slot or NULL
    int tl_wait;
    __device__ __forceinline__ int lane() const { return threadIdx.x; }
    __device__ __forceinline__ int width() const { return PAW_THREADS; }
    __device__ __forceinline__ double sum(double x) const
    {
        const double v = warp_sum(x);
        __syncthreads();                                      // the scratch of the previous reduction has been read
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
        __syncthreads();
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < PAW_THREADS / 32; ++w) s += red[w];
        return s;
    }
    __device__ __forceinline__ bool all(bool b) const { return __syncthreads_and(b ? 1 : 0) != 0; }
    __device__ __forceinline__ int min_int(int x) const
    {
        const int v = __reduce_min_sync(0xffffffffu, x);
        __syncthreads();
        if ((threadIdx.x & 31) == 0) ired[threadIdx.x >> 5] = v;
        __syncthreads();
        int r = ired[0];
#pragma unroll
        for (int w = 1; w < PAW_THREADS / 32; ++w) r = min(r, ired[w]);
        return r;
    }
    __device__ __forceinline__ void sync() const { __syncthreads(); }
    __device__ __forceinline__ void dependency_wait() const
    {
        asm volatile("griddepcontrol.wait;\n" ::: "memory");
        if (tl && threadIdx.x == 0) tl_min(tl, tl_wait);
    }
};

template <int PAW_THREADS, int MINB>
__global__ void __launch_bounds__(PAW_THREADS, MINB) k_propose_wide(ConfigDev cfg, ModelDev m, Level lv, double *bfrag, double *magic, unsigned long long *tl)
{
    __shared__ double red[PAW_THREADS / 32];
    __shared__ int ired[PAW_THREADS / 32];
    pdl_launch_dependents();
    if (threadIdx.x == 0) tl_min(tl, TL_P0);
    const int wi = blockIdx.x;
    const uint32_t e = (uint32_t)lv.order[wi];
    const SweepCtx ctx = lv.ctxs[e >> LV_SLOT_SHIFT];
    const int p = (int)(e & LV_POS_MASK);
    const BlockLanes<PAW_THREADS> co = { red, ired, tl, TL_PW };
    StageSink sink = { m, bfrag, wi, bfrag != nullptr && m.kind == M_MVNORMAL, { 0.0 }, 0.0 };
    propose_particle(co, cfg, m, ctx, p, sink);
    if (!bfrag) { if (threadIdx.x == 0) tl_max(tl, TL_P1); return; }
    double msq = sink.msq;
    if (!sink.on) {
        __syncthreads();                                          // the proposal is complete in global memory
        const double *theta = ctx.prop_theta + (size_t)p * cfg.d;
        msq = 0.0;
        for (int k = threadIdx.x; k < m.ssd_k; k += PAW_THREADS) {
            const double v = centred_mean(m, theta, k);
            msq += v * v;
            bfrag[bfrag_index(m, wi, k)] = v;
        }
    }
    msq = co.sum(msq);
    if (threadIdx.x < 32) stage_scale(m, msq, wi, magic, ctx.ll_acc + p, ctx.ll_q + p, ctx.prop_msq + p);
    if (threadIdx.x == 0) { tl_max(tl, TL_P1); if (tl && wi == 0) tl[TL_N] = (unsigned long long)lv.n; }
}

template <int PAW_THREADS, int MINB, bool TEMPER>
__global__ void __launch_bounds__(PAW_THREADS, MINB) k_accept_wide(ConfigDev cfg, ModelDev m, Level lv, unsigned long long *tl)
{
    __shared__ double red[PAW_THREADS / 32];
    __shared__ int ired[PAW_THREADS / 32];
    pdl_launch_dependents();
    if (threadIdx.x == 0) tl_min(tl, TL_A0);
    const uint32_t e = (uint32_t)lv.order[blockIdx.x];
    const SweepCtx ctx = lv.ctxs[e >> LV_SLOT_SHIFT];
    const BlockLanes<PAW_THREADS> co = { red, ired, tl, TL_AW };
    accept_particle<BlockLanes<PAW_THREADS>, TEMPER>(co, cfg, m, ctx, (int)(e & LV_POS_MASK));
    if (threadIdx.x == 0) tl_max(tl, TL_A1);
}

// ---- the one-pass wide proposal (d <= 4 x 256) ---------------------------------------------------------------------------
// k_propose_wide walks the parameter vector three times (proposal, priors that read another parameter, staging of the
// likelihood kernel's operands), re-reading its own stores from L2 between block-wide barriers, one element per thread and
// trip: on configs[3] a CTA alone on its SM spends 12.6 us behind the dependency wait (profiles/r02_c4_timeline*.txt), and
// that latency x 4 resident CTAs per SM is the throughput of the level.  Here every thread owns FOUR elements
// (k = tid + 256 i) for the whole kernel: all their loads are issued together, the proposal values stay in registers for
// the prior and the staging, the first four elements of the vector (where the hyper-parameters a NORMAL_REF prior or the
// hierarchical mean refer to live) are broadcast through shared memory, and ONE combined reduction ends the kernel.  Two
// neighbouring threads share each Philox call of the noise and kappa draws (two uniforms per call) through a shuffle.
// Same per-element arithmetic as de_particle.h; only the order of the block-wide sums differs.
constexpr int PW1_T = 256, PW1_E = 4;

__device__ __forceinline__ double shfl_xor1(double v)
{
    return __hiloint2double(__shfl_xor_sync(0xffffffffu, __double2hiint(v), 1), __shfl_xor_sync(0xffffffffu, __double2loint(v), 1));
}

template <int MINB>
__global__ void __launch_bounds__(PW1_T, MINB) k_propose_wide1(ConfigDev cfg, ModelDev m, Level lv, double *__restrict__ bfrag, double *magic, unsigned long long *tl)
{
    constexpr int T = PW1_T, E = PW1_E, NW = T / 32;
    __shared__ double red[NW];
    __shared__ int ired[NW];
    __shared__ double red4[NW][4];
    __shared__ double s_head[4], s_headlog[4];
    pdl_launch_dependents();
    const int tid = threadIdx.x;
    if (tid == 0) tl_min(tl, TL_P0);
    const int wi = blockIdx.x;
    const uint32_t e = (uint32_t)lv.order[wi];
    const SweepCtx ctx = lv.ctxs[e >> LV_SLOT_SHIFT];
    const int p = (int)(e & LV_POS_MASK);
    const BlockLanes<T> co = { red, ired, tl, TL_PW };
    const int Np = cfg.Np, d = cfg.d;
    const int g = p / Np, j = p - g * Np;
    const uint32_t unit = (uint32_t)((cfg.group_begin + g) * Np + j);
    const bool replay = ctx.replay != 0;
    const uint32_t sweep = ctx.sweep;

    int kind, i0 = -1, i1 = -1, i2 = -1, hr0 = -1, hr1 = -1, hr2 = -1;
    double g1 = 0.0, g2 = 0.0, u_base = 0.0;
    if (replay) {
        kind = ctx.t_kind[p];
        i0 = ctx.t_idx[p * 3]; i1 = ctx.t_idx[p * 3 + 1]; i2 = ctx.t_idx[p * 3 + 2];
        if (cfg.resample) { hr0 = ctx.t_idx_row[p * 3]; hr1 = ctx.t_idx_row[p * 3 + 1]; hr2 = ctx.t_idx_row[p * 3 + 2]; }
        g1 = ctx.t_g1[p]; g2 = ctx.t_g2[p];
    } else {
        const PlanRec pl = ctx.plan ? load_plan(ctx.plan + p) : make_plan(cfg, ctx, p);
        kind = pl.kind; i0 = pl.i0; i1 = pl.i1; i2 = pl.i2; hr0 = pl.hr0; hr1 = pl.hr1; hr2 = pl.hr2; u_base = pl.u_base; g1 = pl.g1; g2 = pl.g2;
    }
    const bool is_mut = kind == KIND_MUTATION;
    const int block = ctx.block;
    const uint8_t *mask = (block >= 0 && !is_mut) ? cfg.blocks + (size_t)block * d : nullptr;
    const bool use_kappa = !is_mut && cfg.kappa != 1.0;

    // state-independent inputs of the four elements: live flags, noise, kappa draws.  Element k = tid + T i belongs to the
    // Philox pair k >> 1, which this thread shares with thread tid ^ 1: the even thread draws the pairs of i = 0, 2, the odd
    // one those of i = 1, 3, and each hands the other its half.
    unsigned live = 0;
    double nz[E];
    unsigned keep = 0;
#pragma unroll
    for (int i = 0; i < E; ++i) {
        const int k = tid + T * i;
        nz[i] = 0.0;
        if (k < d && (!mask || mask[k] != 0)) live |= 1u << i;
    }
    if (replay) {
#pragma unroll
        for (int i = 0; i < E; ++i) {
            const int k = tid + T * i;
            if ((live >> i) & 1u) {
                nz[i] = ctx.t_noise[(size_t)p * d + k];
                if (use_kappa && ctx.t_keep[(size_t)p * d + k] != 0) keep |= 1u << i;
            }
        }
    } else {
        const unsigned live_pair = live | __shfl_xor_sync(0xffffffffu, live, 1);
#pragma unroll
        for (int i = 0; i < E; ++i) {
            const int k = tid + T * i;
            const bool mine = ((tid ^ i) & 1) == 0;                       // this thread draws the pair of trip i
            dbl2 z; z.a = 0.0; z.b = 0.0;
            unsigned kp = 0;
            if (mine && ((live_pair >> i) & 1u)) {
                const dbl2 u = uniform2(cfg.seed, ST_NOISE, sweep, unit, (uint32_t)(k >> 1));
                if (is_mut) z = normal2(u, cfg.sigma);
                else { z.a = -cfg.eps + (cfg.eps - (-cfg.eps)) * u.a; z.b = -cfg.eps + (cfg.eps - (-cfg.eps)) * u.b; }
                if (use_kappa) {
                    const dbl2 uk = uniform2(cfg.seed, ST_KAPPA, sweep, unit, (uint32_t)(k >> 1));
                    kp = (uk.a <= (1.0 - cfg.kappa) ? 1u : 0u) | (uk.b <= (1.0 - cfg.kappa) ? 2u : 0u);
                }
            }
            // the drawer keeps the half of its own parity and sends the other one
            const double give = (tid & 1) ? z.a : z.b, got = shfl_xor1(give);
            const unsigned kgot = __shfl_xor_sync(0xffffffffu, kp, 1);
            const double own = (tid & 1) ? z.b : z.a;
            const unsigned kbit = ((mine ? kp : kgot) >> (tid & 1)) & 1u;
            if ((live >> i) & 1u) { nz[i] = mine ? own : got; if (kbit) keep |= 1u << i; }
        }
    }
    co.dependency_wait();

    const double *__restrict__ tcur = ctx.cur_theta + (size_t)p * d;
    double *__restrict__ prop = ctx.prop_theta + (size_t)p * d;
    const size_t gbase = (size_t)g * Np;
    const size_t P_all = (size_t)cfg.P_hist;
#define DE_SLOT(k) (((k) < j ? ctx.next_theta : ctx.cur_theta) + (gbase + (size_t)(k)) * d)
#define DE_HIST(r, id) (ctx.hist_theta + ((size_t)(r) * P_all + (size_t)ctx.hist_pos[(size_t)(r) * P_all + (size_t)(id)]) * d)
#define DE_DONOR(k, r) (cfg.resample ? DE_HIST(r, k) : DE_SLOT(k))
    double r1 = 0.0, r2 = 0.0;
    const double *__restrict__ pm = nullptr, *__restrict__ pn = nullptr, *__restrict__ px = nullptr;     // px: the base (DE) or z (snooker)
    bool has_base = false;
    double t[E];
#pragma unroll
    for (int i = 0; i < E; ++i) { const int k = tid + T * i; t[i] = k < d ? tcur[k] : 0.0; }
    if (kind == KIND_DE) {
        pm = DE_DONOR(i1, hr1); pn = DE_DONOR(i2, hr2);
        has_base = cfg.proposal == 0 && ctx.in_burnin != 0;
        if (has_base) {
            if (ctx.exact_base) px = DE_SLOT(i0);
            else {
                const double *cw = ctx.base_cw + gbase;
                const double tt = u_base * ctx.base_tot[g];
                int found = Np - 1;
                for (int q0 = 0; q0 < Np - 1; q0 += T) {
                    const int q = q0 + tid;
                    const bool hit = q < Np - 1 && !(cw[q] < tt);
                    const int best = co.min_int(hit ? q : 0x7fffffff);
                    if (best != 0x7fffffff) { found = best; break; }
                }
                px = ctx.cur_theta + (gbase + (size_t)found) * d;
            }
        }
    } else if (kind == KIND_SNOOKER) {
        px = DE_DONOR(i0, hr0); pm = DE_DONOR(i1, hr1); pn = DE_DONOR(i2, hr2);
        double v1m = 0.0, v1n = 0.0, v2 = 0.0;
#pragma unroll
        for (int i = 0; i < E; ++i) {
            const int k = tid + T * i;
            if (k < d) {
                const double pd = sub(t[i], px[k]);
                v1m = add(v1m, mul(pm[k], pd));
                v1n = add(v1n, mul(pn[k], pd));
                v2 = add(v2, mul(pd, pd));
            }
        }
        v1m = co.sum(v1m); v1n = co.sum(v1n); v2 = co.sum(v2);
        r1 = v1m / v2; r2 = v1n / v2;
    }
#undef DE_DONOR
#undef DE_HIST
#undef DE_SLOT

    if (tid == 0) tl_max(tl, TL_Q0);
    // the proposal: every load first, then the arithmetic and the stores
    double a[E], b[E], c[E];
#pragma unroll
    for (int i = 0; i < E; ++i) {
        const int k = tid + T * i;
        a[i] = 0.0; b[i] = 0.0; c[i] = 0.0;
        if (k < d && !is_mut) {
            if ((live >> i) & 1u) { a[i] = pm[k]; b[i] = pn[k]; }
            if (kind == KIND_SNOOKER || (has_base && ((live >> i) & 1u))) c[i] = px[k];
        }
    }
    double v[E];
    double sq1 = 0.0, sq2 = 0.0;
#pragma unroll
    for (int i = 0; i < E; ++i) {
        const int k = tid + T * i;
        v[i] = 0.0;
        if (k >= d) continue;
        const bool lv_ = (live >> i) & 1u;
        double x;
        if (!lv_) x = t[i];
        else if (is_mut) x = add(t[i], nz[i]);
        else if (kind == KIND_DE) x = de_elem(t[i], a[i], b[i], has_base ? c[i] : t[i], g1, g2, has_base, nz[i]);
        else x = snooker_elem(t[i], c[i], r1, r2, g1, nz[i]);
        if (lv_ && ((keep >> i) & 1u)) x = t[i];                              // recombination! (crossover.jl:301-321)
        if (kind == KIND_SNOOKER) {                                            // adjust_loglike (crossover.jl:268-273)
            const double aa = sub(x, c[i]), bb = sub(t[i], c[i]);
            sq1 = add(sq1, mul(aa, aa)); sq2 = add(sq2, mul(bb, bb));
        }
        v[i] = x;
        prop[k] = x;
        if (ctx.tr_theta) ctx.tr_theta[(size_t)p * d + k] = x;
    }
    // (the logarithm a NORMAL_REF prior needs of its sd parameter: once, by the thread that owns the parameter, not by
    // every warp after the barrier; only when some prior refers to another parameter)
    if (tid < 4) { s_head[tid] = v[0]; s_headlog[tid] = m.prior_has_ref ? log(v[0]) : 0.0; }
    __syncthreads();
    if (tid == 0) tl_max(tl, TL_Q1);

    // bounds, priors and the staging of the likelihood kernel's operands, from the registers
    const bool stage_hier = bfrag != nullptr && m.kind == M_HIER, stage_mvn = bfrag != nullptr && m.kind == M_MVNORMAL;
    const double head0 = s_head[0];
    bool ok = true;
    double ps = 0.0, msq = 0.0;
    double ref_sd = qnan(), ref_log = 0.0;
    // every element's bounds, prior kind and first parameter are fetched before any of them is used (a loop that branches
    // on the kind it has just loaded runs its four L2 round trips one after the other: 4.4 us of the 8.9 a lone CTA spent
    // behind the dependency wait); the remaining parameters are only read for the kinds that need them
    {
        double lo[E], hi[E], pa[E];
        int2 kr[E];
#pragma unroll
        for (int i = 0; i < E; ++i) {
            const int k = min(tid + T * i, d - 1);
            lo[i] = cfg.lo[k]; hi[i] = cfg.hi[k];
            kr[i] = *reinterpret_cast<const int2 *>(&m.prior[k].kind);          // kind, ref
            pa[i] = m.prior[k].a;
        }
#pragma unroll
        for (int i = 0; i < E; ++i) {
            const int k = tid + T * i;
            if (k >= d) continue;
            const double x = v[i];
            ok = ok && (x >= lo[i] && x <= hi[i]);
            if (kr[i].x == PRIOR_NORMAL_REF) {
                const double sd = kr[i].y < 4 ? s_head[kr[i].y] : prop[kr[i].y];
                if (!(sd == ref_sd)) { ref_sd = sd; ref_log = kr[i].y < 4 ? s_headlog[kr[i].y] : log(sd); }
                const double z = (x - pa[i]) / sd;
                ps += -(z * z + DE_LOG2PI) / 2.0 - ref_log;
            } else if (kr[i].x != PRIOR_FLAT) ps += prior_elem(m.prior[k], x, 0.0);
            else ps += 0.0;
        }
    }
    if (tid == 0) tl_max(tl, TL_Q2);
    if (stage_hier || stage_mvn) {
        const int shift = stage_hier ? 2 : 0;                                 // dimension kk of the likelihood is element kk + shift
        double *__restrict__ bf_row = bfrag + bfrag_base(m, wi);
        double cen[E];
#pragma unroll
        for (int i = 0; i < E; ++i) { const int kk = tid + T * i - shift; cen[i] = (kk >= 0 && kk < m.ssd_k) ? m.center[kk] : 0.0; }
#pragma unroll
        for (int i = 0; i < E; ++i) {
            const int kk = tid + T * i - shift;
            if (kk < 0 || kk >= m.ssd_k) continue;
            const double cm = stage_hier ? (head0 + v[i]) - cen[i] : v[i] - cen[i];
            msq += cm * cm;
            bf_row[bfrag_offset(m, wi % SSD_OCT, kk)] = cm;
        }
    }
    const bool inb = __syncthreads_and(ok ? 1 : 0) != 0;
    if (tid == 0) tl_max(tl, TL_Q3);
    ps = warp_sum(ps); msq = warp_sum(msq);
    if (kind == KIND_SNOOKER) { sq1 = warp_sum(sq1); sq2 = warp_sum(sq2); }
    if ((tid & 31) == 0) { red4[tid >> 5][0] = ps; red4[tid >> 5][1] = msq; red4[tid >> 5][2] = sq1; red4[tid >> 5][3] = sq2; }
    __syncthreads();
    if (tid == 0) {
        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll
        for (int w = 0; w < NW; ++w) { s0 += red4[w][0]; s1 += red4[w][1]; s2 += red4[w][2]; s3 += red4[w][3]; }
        ctx.prop_prior[p] = s0;
        ctx.prop_inb[p] = inb ? 1 : 0;
        ctx.prop_adj[p] = kind == KIND_SNOOKER ? adjust_loglike(s2, s3, d) : 0.0;
        if (bfrag) stage_scale(m, s1, wi, magic, ctx.ll_acc + p, ctx.ll_q + p, ctx.prop_msq + p);
        tl_max(tl, TL_P1);
        if (tl && wi == 0) tl[TL_N] = (unsigned long long)lv.n;
    }
}

// DEMCMC_WIDE_SHAPE=<accept digit><propose digit> (A/B runs, tests).  Accept: 0 = 256 threads x 4 CTAs per SM, else 128 x 12 (40 registers, no spills).
// Propose: 0 = the three-pass kernel at 256 x 4, 2 = at 128 x 8, 5 = the one-pass kernel (also tried: 256 x 6, 128 x 12, 64 x 16: slower)
// Measured on configs[3] (M updates/s, 60 iterations):
// 00: 16.6, 22: 17.5, 32: 17.9 (19.3 with the threaded planner), 35: 20.9 -> 21.7 (prior loads hoisted, cheap staging index); the one-pass kernel at 3 / 2 CTAs per SM (80 / 116 registers): 19.9 / 17.1, at 5 / 6 CTAs per SM (48 / 40 registers, 470 / 850 B of spills): 23.8 / 21.3 against 25.0
static int wide_shape()
{
    const char *e = getenv("DEMCMC_WIDE_SHAPE");
    return e ? atoi(e) : 35;
}
static bool wide_enabled(const ConfigDev &cfg)
{
    const char *e = getenv("DEMCMC_NO_WIDE");
    return cfg.d >= PAW_MIN_D && !(e && e[0] == '1');
}

int launch_propose(const ConfigDev &cfg, const ModelDev &m, const Level &lv)
{
    const int blocks = (lv.n * 32 + PA_THREADS - 1) / PA_THREADS;
    XdStage *xs = nullptr;
    if (is_ssd(m.kind)) {
        // sized once for the handle's whole population so it never grows inside a run
        xs = xd_stage(m, std::max(lv.n, cfg.G_local * cfg.Np));
        if (!xs) return -1;
    }
    if (wide_enabled(cfg) && lv.ctxs) {
        // 256 threads, 4 CTAs per SM (64 registers, a few spills): measured on configs[3] against
        // 2 / 3 CTAs per SM and 512 threads x 1 / 2: 14.9 vs 12.7 / 14.0 / 10.8 / 13.5 M updates/s
        double *bf = xs ? xs->bfrag : nullptr, *mg = xs ? xs->magic : nullptr;
        if (cfg.d <= PW1_T * PW1_E && m.kind != M_MVN_FULL && wide_shape() % 10 >= 5) {
            CU(launch_chained(k_propose_wide1<4>, dim3(lv.n), dim3(PW1_T), 0, cfg, m, lv, bf, mg, tl_slot()));
            LAUNCHED("k_propose_wide1");
            return 0;
        }
        switch (wide_shape() % 10) {
        case 2: CU(launch_chained(k_propose_wide<128, 8>, dim3(lv.n), dim3(128), 0, cfg, m, lv, bf, mg, tl_slot())); break;
        default: CU(launch_chained(k_propose_wide<256, 4>, dim3(lv.n), dim3(256), 0, cfg, m, lv, bf, mg, tl_slot())); break;
        }
        LAUNCHED("k_propose_wide");
        return 0;
    }
    CU(launch_chained(k_propose, dim3(blocks), dim3(PA_THREADS), 0, cfg, m, lv, xs ? xs->bfrag : nullptr, xs ? xs->magic : nullptr, tl_slot()));
    LAUNCHED("k_propose");
    return 0;
}

int launch_accept(const ConfigDev &cfg, const ModelDev &m, const Level &lv)
{
    const int blocks = (lv.n * 32 + PA_THREADS - 1) / PA_THREADS;
    if (wide_enabled(cfg) && lv.ctxs) {
        switch (wide_shape() / 10) {
        case 0: CU(cfg.temp ? launch_chained(k_accept_wide<256, 4, true>, dim3(lv.n), dim3(256), 0, cfg, m, lv, tl_slot())
                            : launch_chained(k_accept_wide<256, 4, false>, dim3(lv.n), dim3(256), 0, cfg, m, lv, tl_slot())); break;
        default: CU(cfg.temp ? launch_chained(k_accept_wide<128, 12, true>, dim3(lv.n), dim3(128), 0, cfg, m, lv, tl_slot())
                             : launch_chained(k_accept_wide<128, 12, false>, dim3(lv.n), dim3(128), 0, cfg, m, lv, tl_slot())); break;
        }
        LAUNCHED("k_accept_wide");
        if (g_tl_cap > 0) ++g_tl_level;
        return 0;
    }
    if (cfg.temp) CU(launch_chained(k_accept<true>, dim3(blocks), dim3(PA_THREADS), 0, cfg, m, lv, tl_slot()));
    else CU(launch_chained(k_accept<false>, dim3(blocks), dim3(PA_THREADS), 0, cfg, m, lv, tl_slot()));
    LAUNCHED("k_accept");
    if (g_tl_cap > 0) ++g_tl_level;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// select_base preparation (crossover.jl:282-289) on the sweep-start weights, one block per group:
// theta = exp.(w)/sum(exp.(w)); NaN anywhere => the raw weights; running sums for the cumulative walk
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_base_prep(ConfigDev cfg, const double *w, double *th, double *cw, double *tot)
{
    const int g = blockIdx.x, Np = cfg.Np;
    const double *wg = w + (size_t)g * Np;
    double *tg = th + (size_t)g * Np, *cg = cw + (size_t)g * Np;
    __shared__ double s_tot;
    for (int i = threadIdx.x; i < Np; i += blockDim.x) tg[i] = exp(wg[i]);
    __syncthreads();
    if (threadIdx.x == 0) { ksum_t k = { 0.0, 0.0 }; for (int i = 0; i < Np; ++i) kadd(k, tg[i]); s_tot = kval(k); }
    __syncthreads();
    bool bad = false;
    for (int i = threadIdx.x; i < Np; i += blockDim.x) { const double v = tg[i] / s_tot; tg[i] = v; bad |= (v != v); }
    const int any_bad = __syncthreads_or(bad ? 1 : 0);
    if (threadIdx.x == 0) {
        const double *src = any_bad ? wg : tg;
        ksum_t k = { 0.0, 0.0 };
        for (int i = 0; i < Np; ++i) kadd(k, src[i]);
        tot[g] = kval(k);
        double c = src[0];
        cg[0] = c;
        for (int i = 1; i < Np; ++i) { c += src[i]; cg[i] = c; }
    }
}

int launch_base_prep(const ConfigDev &cfg, const double *w, double *th, double *cw, double *tot)
{
    k_base_prep<<<cfg.G_local, 128, 0, stream()>>>(cfg, w, th, cw, tot);
    LAUNCHED("k_base_prep");
    return 0;
}

// ------------------------------------------------------------------------------------------------
// the state-independent draws of a whole chunk (de_types.h: PlanRec), one thread per (sweep, particle)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_plan(ConfigDev cfg, const SweepCtx *ctxs, int n_sw, int P)
{
    const int t = blockIdx.x * 128 + threadIdx.x;
    if (t >= n_sw * P) return;
    const int s = t / P, p = t - s * P;
    const SweepCtx &ctx = ctxs[s];
    if (ctx.plan) ctx.plan[p] = make_plan(cfg, ctx, p);
}

int launch_plan(const ConfigDev &cfg, const SweepCtx *d_ctxs, int n_sw)
{
    const int P = cfg.G_local * cfg.Np;
    k_plan<<<(n_sw * P + 127) / 128, 128, 0, stream()>>>(cfg, d_ctxs, n_sw, P);
    LAUNCHED("k_plan");
    g_break_chain = true;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// pointwise likelihood kernels: block = PW_TP particles x one observation split
// ------------------------------------------------------------------------------------------------
// a particle's parameters (+ per-particle constants) as the per-observation densities want them
template <int KIND>
__device__ __forceinline__ void pointwise_par(const ModelDev &m, const double *th, double *par)
{
    if (KIND == M_GAUSSIAN) { par[0] = th[0]; par[1] = th[1]; par[2] = log(th[1]); }
    else if (KIND == M_LNR) { for (int r = 0; r <= m.n_dim; ++r) par[r] = th[r]; }
    else {
        double pneg = 1.0;
        for (int r = 0; r < m.n_dim; ++r) { par[r] = th[r]; pneg *= norm_cdf(-th[r]); }
        par[m.n_dim] = th[m.n_dim]; par[m.n_dim + 1] = th[m.n_dim + 1]; par[m.n_dim + 2] = th[m.n_dim + 2];
        par[m.n_dim + 3] = 1.0 / (1.0 - pneg);
        par[m.n_dim + 4] = 1.0 / th[m.n_dim];
    }
}

// Small pointwise problems (the reference's own examples and tests: tens of observations, a handful
// of particles per group): the whole update of a particle -- proposal, likelihood over all
// observations, accept -- by ONE warp in ONE launch per level.  The three-kernel chain of a level
// costs ~13 us of launches and hand-offs, which is all there is to do on configs[0].
struct NoWaitLanes : WarpLanes { __device__ __forceinline__ void dependency_wait() const {} };
// the whole update of one particle by one warp (small pointwise problems, n_split == 1): C = WarpLanes inside a PDL chain,
// NoWaitLanes where the caller has done the waiting
template <int KIND, bool TEMPER, class C>
__device__ __forceinline__ void fused_update(const C &co, const ConfigDev &cfg, const ModelDev &m, const SweepCtx &ctx, int p)
{
    const int lane = threadIdx.x & 31;
    NullSink sink;
    propose_particle(co, cfg, m, ctx, p, sink);
    __syncwarp();
    if (KIND == M_GAUSSIAN || KIND == M_LNR || KIND == M_LBA) {
        double par[MAX_ACC + 5];
        pointwise_par<KIND>(m, ctx.prop_theta + (size_t)p * cfg.d, par);
        const double *sg = m.has_sigma ? m.sigma_acc : nullptr;
        double a = 0.0;
        for (int64_t i = lane; i < m.n_obs; i += 32) {
            const double x = m.x[i];
            if (KIND == M_GAUSSIAN) a += gaussian_obs(par, x);
            else if (KIND == M_LNR) a += lnr_obs(par, m.n_dim, sg, x, m.choice[i] - 1);
            else a += lba_obs(par, m.n_dim, par[m.n_dim + 3], m.lba_floor, x, m.choice[i] - 1);
        }
        a = warp_sum(a);
        if (lane == 0) ctx.ll_part[(size_t)p] = a;               // n_split == 1 on this path
        __syncwarp();
    }
    accept_particle<NoWaitLanes, TEMPER>(NoWaitLanes(), cfg, m, ctx, p);
}

// TEMPER (here, in k_chunk_small and k_accept_wide): as k_accept's
template <int KIND, bool TEMPER>
__global__ void __launch_bounds__(PA_THREADS) k_level_fused(ConfigDev cfg, ModelDev m, Level lv)
{
    pdl_launch_dependents();
    const int wi = (blockIdx.x * PA_THREADS + threadIdx.x) >> 5;
    if (wi >= lv.n) { pdl_wait(); return; }
    const uint32_t e = (uint32_t)lv.order[wi];
    const SweepCtx ctx = lv.ctxs[e >> LV_SLOT_SHIFT];
    fused_update<KIND, TEMPER>(WarpLanes(), cfg, m, ctx, (int)(e & LV_POS_MASK));
}

// The reference's own examples (Gaussian_Example.jl: 4 groups x 6 particles, 50 observations) are a handful of warps: a
// launch per dependency level -- ~8 us each, 3.7 per sweep -- is all there is to their step.  When the whole population
// fits one CTA, ONE launch runs every level of a chunk (up to 16 sweeps): a warp per update, a block-wide barrier between
// levels (the state rows are global memory written and read by the same SM).
constexpr int SC_MAX_LEVELS = 640, SC_MAX_WARPS = 12;       // 12 warps x 168 registers fit one SM
constexpr int SC_MAX_P = 96;                                // beyond, a level is several rounds of the 12 warps and the level-by-level path (all SMs) wins
struct SmallChunk { int32_t n_levels; int32_t off[SC_MAX_LEVELS + 1]; };
template <int KIND, bool TEMPER>
__global__ void __launch_bounds__(SC_MAX_WARPS * 32, 1) k_chunk_small(const __grid_constant__ ConfigDev cfg, const __grid_constant__ ModelDev m,
                                                                       const int32_t *order, const SweepCtx *ctxs, const __grid_constant__ SmallChunk sc)
{
    const int warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int L = 0; L < sc.n_levels; ++L) {
        for (int wi = sc.off[L] + warp; wi < sc.off[L + 1]; wi += nw) {
            const uint32_t e = (uint32_t)order[wi];
            const SweepCtx ctx = ctxs[e >> LV_SLOT_SHIFT];
            fused_update<KIND, TEMPER>(NoWaitLanes(), cfg, m, ctx, (int)(e & LV_POS_MASK));
        }
        __syncthreads();
    }
}
constexpr int64_t FUSED_MAX_OBS = 256;

// small pointwise models: one warp per update.  DEMCMC_NO_FUSED=1 turns that off, read per call (A/B runs in one process)
static bool fused_eligible(const ConfigDev &cfg, const ModelDev &m)
{
    const char *env = getenv("DEMCMC_NO_FUSED");
    if (env && env[0] == '1') return false;
    if (is_ssd(m.kind) || cfg.d > 64) return false;
    if ((m.kind == M_GAUSSIAN || m.kind == M_LNR || m.kind == M_LBA) && (m.n_obs > FUSED_MAX_OBS || m.n_osplit * m.n_ksplit != 1)) return false;
    return m.kind == M_GAUSSIAN || m.kind == M_LNR || m.kind == M_LBA || m.kind == M_BINOMIAL || m.kind == M_RASTRIGIN;
}

// returns 1 when the level is not a small pointwise one (the caller launches the three kernels)
int launch_level_fused(const ConfigDev &cfg, const ModelDev &m, const Level &lv)
{
    if (!lv.ctxs || !fused_eligible(cfg, m)) return 1;
    const int blocks = (lv.n * 32 + PA_THREADS - 1) / PA_THREADS;
    switch (m.kind) {
    case M_GAUSSIAN: CU(cfg.temp ? launch_chained(k_level_fused<M_GAUSSIAN, true>, dim3(blocks), dim3(PA_THREADS), 0, cfg, m, lv)
                                : launch_chained(k_level_fused<M_GAUSSIAN, false>, dim3(blocks), dim3(PA_THREADS), 0, cfg, m, lv)); break;
    case M_LNR: CU(cfg.temp ? launch_chained(k_level_fused<M_LNR, true>, dim3(blocks), dim3(PA_THREADS), 0, cfg, m, lv)
                                : launch_chained(k_level_fused<M_LNR, false>, dim3(blocks), dim3(PA_THREADS), 0, cfg, m, lv)); break;
    case M_LBA: CU(cfg.temp ? launch_chained(k_level_fused<M_LBA, true>, dim3(blocks), dim3(PA_THREADS), 0, cfg, m, lv)
                                : launch_chained(k_level_fused<M_LBA, false>, dim3(blocks), dim3(PA_THREADS), 0, cfg, m, lv)); break;
    case M_BINOMIAL: CU(cfg.temp ? launch_chained(k_level_fused<M_BINOMIAL, true>, dim3(blocks), dim3(PA_THREADS), 0, cfg, m, lv)
                                : launch_chained(k_level_fused<M_BINOMIAL, false>, dim3(blocks), dim3(PA_THREADS), 0, cfg, m, lv)); break;
    case M_RASTRIGIN: CU(cfg.temp ? launch_chained(k_level_fused<M_RASTRIGIN, true>, dim3(blocks), dim3(PA_THREADS), 0, cfg, m, lv)
                                : launch_chained(k_level_fused<M_RASTRIGIN, false>, dim3(blocks), dim3(PA_THREADS), 0, cfg, m, lv)); break;
    default: return 1;
    }
    LAUNCHED("k_level_fused");
    if (g_tl_cap > 0) ++g_tl_level;
    return 0;
}

// returns 1 when the chunk is not a small pointwise one (the caller launches level by level)
int launch_chunk_small(const ConfigDev &cfg, const ModelDev &m, const int32_t *d_order, const SweepCtx *d_ctx, const int32_t *level_off, int n_levels)
{
    const char *env = getenv("DEMCMC_NO_SMALL");
    if ((env && env[0] == '1') || !fused_eligible(cfg, m)) return 1;
    if (n_levels <= 0 || n_levels > SC_MAX_LEVELS || cfg.G_local * cfg.Np > SC_MAX_P) return 1;
    SmallChunk sc;
    sc.n_levels = n_levels;
    int widest = 1;
    for (int l = 0; l <= n_levels; ++l) sc.off[l] = level_off[l];
    for (int l = 0; l < n_levels; ++l) widest = std::max(widest, level_off[l + 1] - level_off[l]);
    const int threads = 32 * std::min(widest, SC_MAX_WARPS);
    auto go = [&](auto kernel_untempered, auto kernel_tempered) {
        if (cfg.temp) kernel_tempered<<<1, threads, 0, stream()>>>(cfg, m, d_order, d_ctx, sc);
        else kernel_untempered<<<1, threads, 0, stream()>>>(cfg, m, d_order, d_ctx, sc);
    };
    switch (m.kind) {
    case M_GAUSSIAN: go(k_chunk_small<M_GAUSSIAN, false>, k_chunk_small<M_GAUSSIAN, true>); break;
    case M_LNR: go(k_chunk_small<M_LNR, false>, k_chunk_small<M_LNR, true>); break;
    case M_LBA: go(k_chunk_small<M_LBA, false>, k_chunk_small<M_LBA, true>); break;
    case M_BINOMIAL: go(k_chunk_small<M_BINOMIAL, false>, k_chunk_small<M_BINOMIAL, true>); break;
    default: go(k_chunk_small<M_RASTRIGIN, false>, k_chunk_small<M_RASTRIGIN, true>); break;
    }
    LAUNCHED("k_chunk_small");
    if (g_tl_cap > 0) g_tl_level += n_levels;
    return 0;
}

template <int KIND>
__global__ void __launch_bounds__(PW_THREADS) k_ll_pointwise(ModelDev m, const double *theta, Level lv, double *part)
{
    constexpr int NPAR = MAX_ACC + 5;
    __shared__ double par[PW_TP][NPAR];
    __shared__ double red[PW_THREADS / 32][PW_TP];
    const int tile = blockIdx.x, split = blockIdx.y, tid = threadIdx.x;
    const int nt = min(PW_TP, lv.n - tile * PW_TP);
    const int n_split = m.n_osplit * m.n_ksplit;
    // stage the tile's parameters (+ per-particle constants)
    if (tid < nt) {
        const int p = lv.order ? (int)((uint32_t)lv.order[tile * PW_TP + tid] & LV_POS_MASK) : tile * PW_TP + tid;
        pointwise_par<KIND>(m, theta + (size_t)p * m.d, par[tid]);
    }
    __syncthreads();
    double acc[PW_TP];
#pragma unroll
    for (int t = 0; t < PW_TP; ++t) acc[t] = 0.0;
    const int64_t i0 = (int64_t)split * m.split_len;
    const int64_t i1 = min(m.n_obs, i0 + (int64_t)m.split_len);
    const double *sg = m.has_sigma ? m.sigma_acc : nullptr;
    if (KIND != M_GAUSSIAN) {
        // LNR / LBA: ONE copy of the density in the instruction stream, particles in the outer loop.
        // With the eight particles of the tile unrolled around it the loop body was 108 KB of code and
        // a quarter of the stall samples were instruction fetches (ncu: no_instructions 24 %); the
        // CTA's slice of observations (a few KB) stays in L1 across the particles.  Same summation
        // order per particle as the unrolled form: bit-identical sums.
#pragma unroll 1
        for (int t = 0; t < nt; ++t) {
            double a = 0.0;
            for (int64_t i = i0 + tid; i < i1; i += PW_THREADS) {
                const double x = m.x[i];
                const int c = m.choice[i] - 1;
                if (KIND == M_LNR) a += lnr_obs(par[t], m.n_dim, sg, x, c);
                else a += lba_obs(par[t], m.n_dim, par[t][m.n_dim + 3], m.lba_floor, x, c);
            }
            const double v = warp_sum(a);
            if ((tid & 31) == 0) red[tid >> 5][t] = v;
        }
    } else
    for (int64_t i = i0 + tid; i < i1; i += PW_THREADS) {
        const double x = m.x[i];
        const int c = (KIND == M_GAUSSIAN) ? 0 : m.choice[i] - 1;
#pragma unroll
        for (int t = 0; t < PW_TP; ++t) {
            if (t < nt) {
                if (KIND == M_GAUSSIAN) acc[t] += gaussian_obs(par[t], x);
                else if (KIND == M_LNR) acc[t] += lnr_obs(par[t], m.n_dim, sg, x, c);
                else acc[t] += lba_obs(par[t], m.n_dim, par[t][m.n_dim + 3], m.lba_floor, x, c);
            }
        }
    }
    if (KIND == M_GAUSSIAN) {
#pragma unroll
        for (int t = 0; t < PW_TP; ++t) {
            const double v = warp_sum(acc[t]);
            if ((tid & 31) == 0) red[tid >> 5][t] = v;
        }
    }
    __syncthreads();
    if (tid < nt) {
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < PW_THREADS / 32; ++w) v += red[w][tid];
        const int p = lv.order ? (int)((uint32_t)lv.order[tile * PW_TP + tid] & LV_POS_MASK) : tile * PW_TP + tid;
        part[(size_t)p * n_split + split] = v;
    }
}

// ------------------------------------------------------------------------------------------------
// MVN / hierarchical likelihood kernel.  With centred data x' and centred means m',
//   sum_i sum_k (x_ik - m_pk)^2 = sum x'^2 - 2 B_p + n sum_k m'_pk^2,   B_p = sum_i sum_k x'_ik m'_pk
// and only B_p needs the O(N d) pass: one multiply-add per (observation, dimension, particle), every
// observation streamed for every particle (no sufficient-statistic shortcut).
//
// B = X' M is a GEMM whose rows are summed away, so it runs on the fp64 tensor path: DMMA m8n8k4
// measures 37.1 TFLOP/s on B200 against 33.9 for DFMA (scripts/probes/probe_dmma.cu; the two share
// one pipe, they do not add), and it needs 8x fewer issue slots and no accumulator tile.
//   A (8 observations x 4 dimensions)  = packed centred data, streamed
//   B (4 dimensions x 8 particles)     = centred means of one particle octet, held in REGISTERS for
//                                        the whole kernel (<= 13 k-steps x 4 octets per thread)
//   C (8 observations x 8 particles)   = per-row-pair cross terms; a chain runs over the k-steps
//                                        of ONE observation tile, then is rounded to the
//                                        particle's fixed-point grid (de_math.h: xd_scale) and added
//                                        as an integer, which makes the total independent of how
//                                        observation tiles were dealt to CTAs
// CTA = 4 warps x one particle tile (32 particles = 4 octets).  Warp w owns row pair w (16 of the 64
// observations) of every observation tile in the CTA's range: its operand stream is contiguous in
// the packed layout, so each warp runs a PRIVATE 4-stage ring of TMA bulk copies (cp.async.bulk,
// one copy per stage, completing on the warp's own mbarriers) and the kernel has no CTA-wide
// barrier and no cross-warp wait at all.  Inner step: one LDS.128 (A fragments of two row tiles)
// feeds 8 DMMAs (2 row tiles x 4 octets) on 4 accumulator chains per warp (one per octet; the two
// row tiles of the pair add into the same chain, 4 DMMAs apart, so a tile ends with 8 conversions).
// The launch is one wave: CTAs are dealt to particle tiles in proportion to their octets (the last
// tile of a level may hold 1..4), each taking a balanced contiguous range of observation tiles;
// padding costs at most 7 particles per level.
// ------------------------------------------------------------------------------------------------
constexpr int XD_THREADS = 128;
constexpr int XD_STAGES = 4;
constexpr int XD_CTAS_PER_SM = 2;
constexpr int XD_KPC_MAX_TILES = 8;   // observation streams this short take several dimension splits per CTA (XdGrid::kpc)
constexpr int XD_MIN_TILES = 4;          // observation tiles a CTA should at least stream (amortises its prologue)
constexpr int XD_WAVE_TILES = 48;        // observation tiles per CTA when a level needs several waves

// ---- TMA bulk copy + mbarrier helpers (sm_90+; SASS: UBLKCP / SYNCS) -----------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    // try_wait sleeps in hardware between polls; the bound turns a protocol bug into a trap, not a hang
    for (uint32_t spins = 0; !mbar_try_wait(bar, parity); ++spins)
        if (spins > (1u << 26)) __trap();
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// D(8x8) += A(8x4) * B(4x8) in fp64 on the tensor path (SASS: DMMA.8x8x4)
__device__ __forceinline__ void dmma884(double &c0, double &c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

static size_t xdot_smem_bytes(int nj, int stages = XD_STAGES)
{
    return (size_t)4 * stages * nj * 64 * sizeof(double) + sizeof(uint64_t) * 4 * stages;
}

static size_t xd_bfrag_doubles(const ModelDev &m, int n) { return (size_t)((n + SSD_OCT - 1) / SSD_OCT) * m.n_ksplit * m.ssd_nj * 32; }
static XdStage *xd_stage(const ModelDev &m, int n)
{
    XdStage &x = g_xs[g_dev][g_lane];
    const size_t need = xd_bfrag_doubles(m, n) + (size_t)((n + SSD_OCT - 1) / SSD_OCT) * SSD_OCT;
    if (need > x.cap) {
        cudaStreamSynchronize(stream());
        if (x.bfrag) cudaFree(x.bfrag);
        x.bfrag = nullptr; x.magic = nullptr; x.cap = 0;
        if (cudaMalloc(&x.bfrag, sizeof(double) * need) != cudaSuccess) { g_be_err = "cudaMalloc(mean staging)"; return nullptr; }
        x.cap = need;
    }
    // the dimension slots that pad a split to whole k-steps must read as zero, and the geometry may
    // change with the model: clear whenever the split between the two arrays moves
    double *magic = x.bfrag + (x.cap - (size_t)((n + SSD_OCT - 1) / SSD_OCT) * SSD_OCT);
    // (the staging buffers outlive the handles: another model's layout leaves its means where this one's padding is)
    const long long geom = ((long long)m.ssd_k << 40) ^ ((long long)m.ksplit_len << 24) ^ ((long long)m.n_ksplit << 12) ^ ((long long)m.ssd_nj << 4) ^ (long long)m.ssd_half;
    if (magic != x.magic || geom != x.geom) {
        x.geom = geom;
        if (cudaMemsetAsync(x.bfrag, 0, sizeof(double) * x.cap, stream()) != cudaSuccess) { g_be_err = "cudaMemset(mean staging)"; return nullptr; }
        x.magic = magic;
        x.fresh = true;
    }
    return &x;
}

// how the CTAs of one launch are dealt to the particle tiles of a level
// n_hi tiles of oct_hi octets with c_hi CTAs each, then n_lo tiles of oct_lo octets with c_lo CTAs each
// kpc: dimension splits one CTA walks (1 unless the observation stream is a few tiles long: the hierarchical model with 50
// observations per subject has ONE tile and 20 splits of 52 subjects -- a CTA per (particle tile, split) is all launch
// latency, 1160 CTAs in four waves for a level of 1834 updates; its CTAs take several splits each so the level fits one wave)
struct XdGrid { int32_t n_hi, oct_hi, c_hi, n_lo, oct_lo, c_lo, kpc; };

// Where one warp of k_xdot / k_chunk_persist keeps its operand ring: the warp's index inside its
// 4-warp CTA (= the row pair it owns), the dimension split, the ring and its `full` barriers, and the
// number of stages it has consumed so far (the barriers are initialised once per kernel; stage and
// phase parity follow from the running count, so the persistent kernel carries the ring from one
// item to the next without re-initialising anything).
struct XdWarp { int warp, ks; double *ring; uint64_t *full; uint32_t it_base; };

// NJC: the model's k-steps when known at compile time (13), else 0; HALF: (with NJC) the last k-step is
// a half step (de_types.h: ssd_half); STAGES: depth of the warp's operand ring.
// bsrc / b_oct_stride: the tile's B fragments [octet][k-step][lane] (global staging buffer, or the
// shared-memory copy the persistent kernel's helper warp made); msrc: its 8 magic constants per octet.
// HOOKS: operator()() = wait until the means may be read; after_loads() = they are in registers;
// item_end() = the tile's cross terms have been added to ll_acc.
template <int NOCT, int NJC, bool HALF, int STAGES, class HOOKS>
__device__ __forceinline__ void xdot_body(const ModelDev &m, const double *bsrc, size_t b_oct_stride, const double *msrc, const Level &lv,
                                          long long *ll_acc, int oct0, int T0, int T1, XdWarp &xw, const HOOKS &dependency_wait,
                                          unsigned long long *tl, unsigned long long *tlc, int pre_issued = 0)
{
    const int tid = threadIdx.x, warp = xw.warp, lane = tid & 31, ks = xw.ks;
    const int nj = NJC ? NJC : m.ssd_nj;
    const bool half = NJC ? HALF : (m.ssd_half != 0);
    const int n_tiles = (int)(m.ssd_ld / SSD_TN);
    const uint32_t stage_doubles = (uint32_t)nj * 64, stage_bytes = stage_doubles * (uint32_t)sizeof(double);
    double *ring = xw.ring;
    uint64_t *full = xw.full;
    const uint32_t it_base = xw.it_base;
    const double *src = m.xT + (((size_t)(ks * 4 + warp) * n_tiles + T0) * nj) * 64;

    if (lane == 0) {
#pragma unroll
        for (int s = pre_issued; s < STAGES; ++s)            // (pre_issued: the caller has requested the first tiles already)
            if (T0 + s < T1) {
                const uint32_t st = (it_base + (uint32_t)s) % STAGES;
                mbar_expect_tx(&full[st], stage_bytes);
                bulk_g2s(ring + (size_t)st * stage_doubles, src + (size_t)s * stage_doubles, stage_bytes, &full[st]);
            }
    }
    __syncwarp();
    dependency_wait();                                       // the packed data are constant; the means are not
    if (tid == 0) tl_max(tl, TL_XWAIT);
    if (tlc && tid == 0 && blockIdx.x < TL_CTA_MAX) { tlc[blockIdx.x * 4 + 1] = gtime(); tlc[blockIdx.x * 4 + 3] = (unsigned long long)(T1 - T0) * 10 + NOCT; }

    // this tile's centred means as B fragments, and the particles' fixed-point constants (requested
    // first: a warp's shared-memory loads complete in order, so once the first observation tile has
    // consumed every B fragment the constants have landed too -- that is when after_loads() runs)
    double mg[NOCT][2];
#pragma unroll
    for (int pt = 0; pt < NOCT; ++pt)
#pragma unroll
        for (int e = 0; e < 2; ++e) mg[pt][e] = msrc[pt * SSD_OCT + 2 * (lane & 3) + e];
    double b[SSD_NJ][NOCT];
    {
#pragma unroll
        for (int pt = 0; pt < NOCT; ++pt) {
            // a half step's B fragment repeats its two means in rows 2-3 (de_types.h: ssd_half): the staged
            // fragment holds them once, lanes of rows 2-3 read the slots of rows 0-1
            const double *bf = bsrc + (size_t)pt * b_oct_stride;
#pragma unroll
            for (int j = 0; j < SSD_NJ; ++j) b[j][pt] = j < nj ? bf[j * 32 + ((half && j == nj - 1) ? (lane & ~2) : lane)] : 0.0;
        }
    }
    unsigned long long isum[NOCT][2];
    // one chain per octet (both row tiles of the pair add into it), and TWO sets of them used by
    // alternate observation tiles: a tile's chains are rounded to the fixed-point grid one k-step
    // into the NEXT tile, when they have drained on their own, so the tile boundary costs neither a
    // pipe drain nor a block of conversions
    double accA[NOCT][2], accB[NOCT][2];
#pragma unroll
    for (int pt = 0; pt < NOCT; ++pt)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            isum[pt][e] = 0ull;
            accA[pt][e] = 0.0; accB[pt][e] = 0.0;
        }
    auto convert = [&](double (&acc)[NOCT][2]) {
#pragma unroll
        for (int pt = 0; pt < NOCT; ++pt)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                isum[pt][e] += (unsigned long long)xd_bits(__dadd_rn(acc[pt][e], mg[pt][e]));
                acc[pt][e] = 0.0;
            }
    };
    // one observation tile: its DMMAs go to `acc`; `prev` (the other set) is converted after the
    // first k-step when it holds the previous tile
    auto tile = [&](int t, double (&acc)[NOCT][2], double (&prev)[NOCT][2], bool have_prev, bool first = false) {
        const int it = t - T0;
        const uint32_t gi = it_base + (uint32_t)it, st = gi % STAGES;
        mbar_wait(&full[st], (gi / STAGES) & 1u);
        if (tl && tid == 0 && t == T0) tl_max(tl, TL_XFIRST);
        const double2 *xa = reinterpret_cast<const double2 *>(ring + (size_t)st * stage_doubles) + lane;
        double2 a = xa[0];
#pragma unroll
        for (int j = 0; j < SSD_NJ; ++j) {
            if (j >= nj) break;
            double2 an = a;
            if (j + 1 < nj) an = xa[(j + 1) * 32];
#pragma unroll
            for (int pt = 0; pt < NOCT; ++pt) dmma884(acc[pt][0], acc[pt][1], a.x, b[j][pt]);
            if (!(half && j == nj - 1)) {
#pragma unroll
                for (int pt = 0; pt < NOCT; ++pt) dmma884(acc[pt][0], acc[pt][1], a.y, b[j][pt]);
            }
            a = an;
            if (j == 0 && have_prev) convert(prev);
        }
        __syncwarp();                                        // every lane's reads of the stage have landed
        if (first) dependency_wait.after_loads();            // ... and every B fragment has been an operand of a DMMA
        if (lane == 0 && t + STAGES < T1) {
            mbar_expect_tx(&full[st], stage_bytes);
            bulk_g2s(ring + (size_t)st * stage_doubles, src + (size_t)(it + STAGES) * stage_doubles, stage_bytes, &full[st]);
        }
    };
    int t = T0;
    tile(t++, accA, accB, false, true);
    for (; t + 1 < T1; t += 2) {
        tile(t, accB, accA, true);
        tile(t + 1, accA, accB, true);
    }
    if (t < T1) { tile(t, accB, accA, true); convert(accB); }
    else convert(accA);

    if (tid == 0) { tl_min(tl, TL_XLOOP0); tl_max(tl, TL_XLOOP1); }
    if (tlc && tid == 0 && blockIdx.x < TL_CTA_MAX) tlc[blockIdx.x * 4 + 2] = gtime();
    // remove the magic offsets (one conversion per observation tile), sum the 8 rows held by the
    // lanes of each column group, and add the CTA's share to the particles' accumulators
    const unsigned long long n_conv = (unsigned long long)(T1 - T0);
#pragma unroll
    for (int pt = 0; pt < NOCT; ++pt)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            unsigned long long v = isum[pt][e] - n_conv * (unsigned long long)xd_bits(mg[pt][e]);
#pragma unroll
            for (int o = 4; o < 32; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            const int idx = (oct0 + pt) * SSD_OCT + 2 * lane + e;
            if (lane < 4 && idx < lv.n) {
                const int p = lv.order ? (int)((uint32_t)lv.order[idx] & LV_POS_MASK) : idx;
                atomicAdd(reinterpret_cast<unsigned long long *>(ll_acc) + p, v);
            }
        }
    dependency_wait.item_end();
    if (tid == 0) tl_max(tl, TL_X1);
    xw.it_base = it_base + (uint32_t)(T1 - T0);
}

struct PdlWait {
    __device__ __forceinline__ void operator()() const { pdl_wait(); }
    __device__ __forceinline__ void after_loads() const {}
    __device__ __forceinline__ void item_end() const {}
};

// STAGES / MAXOCT / MINB: <XD_STAGES, 4, XD_CTAS_PER_SM> is the streaming kernel (long observation streams: four-octet tiles, a
// four-stage ring, 252 registers, two CTAs per SM).  <2, 2, 4> serves streams of a few tiles (the hierarchical model's 50
// observations per subject are ONE tile): an item there is all latency -- B-fragment loads, 104 DMMAs, the flush -- so tiles of
// at most two octets at <= 128 registers and a two-stage ring put four CTAs on an SM instead of two.  The DMMA chains (octet,
// row pair, observation tile, dimension split) are the same in both, hence the same fixed-point totals.
template <int STAGES, int MAXOCT, int MINB>
__global__ void __launch_bounds__(XD_THREADS, MINB) k_xdot_t(ModelDev m, const double *bfrag, const double *magic, Level lv,
                                                             long long *ll_acc, XdGrid g, unsigned long long *tl, unsigned long long *tlc)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    pdl_launch_dependents();
    if (threadIdx.x == 0) { tl_min(tl, TL_X0); tl_max(tl, TL_X0MAX); if (tlc && blockIdx.x < TL_CTA_MAX) tlc[blockIdx.x * 4] = gtime(); }
    int oct0, c_in, C, noct;
    const int n_in_hi = g.n_hi * g.c_hi;
    if ((int)blockIdx.x < n_in_hi) { const int t = blockIdx.x / g.c_hi; c_in = blockIdx.x - t * g.c_hi; C = g.c_hi; noct = g.oct_hi; oct0 = t * g.oct_hi; }
    else { const int r = blockIdx.x - n_in_hi, t = r / g.c_lo; c_in = r - t * g.c_lo; C = g.c_lo; noct = g.oct_lo; oct0 = g.n_hi * g.oct_hi + t * g.oct_lo; }
    const int n_tiles = (int)(m.ssd_ld / SSD_TN);
    const int T0 = (int)((int64_t)c_in * n_tiles / C), T1 = (int)((int64_t)(c_in + 1) * n_tiles / C);
    if (T1 <= T0) { pdl_wait(); return; }
    const int warp = threadIdx.x >> 5;
    const uint32_t stage_doubles = (uint32_t)m.ssd_nj * 64;
    XdWarp xw;
    xw.warp = warp; xw.ks = 0; xw.it_base = 0;
    xw.ring = reinterpret_cast<double *>(smem_raw) + (size_t)warp * STAGES * stage_doubles;
    xw.full = reinterpret_cast<uint64_t *>(reinterpret_cast<double *>(smem_raw) + (size_t)4 * STAGES * stage_doubles) + warp * STAGES;
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) mbar_init(&xw.full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    const PdlWait wait;
    const double *msrc = magic + (size_t)oct0 * SSD_OCT;
    const size_t bstride = (size_t)m.n_ksplit * m.ssd_nj * 32;
    const int ks_end = min(m.n_ksplit, ((int)blockIdx.y + 1) * g.kpc);
    // one observation tile per split (<= 64 observations per dimension) and no more splits than ring stages: every split's
    // tile is requested up front, so the later ones arrive while the earlier ones are multiplied
    const bool ahead = n_tiles == 1 && g.kpc > 1 && g.kpc <= STAGES;
    if (ahead && (threadIdx.x & 31) == 0) {
        int i = 0;
        for (int ks = blockIdx.y * g.kpc; ks < ks_end; ++ks, ++i) {
            mbar_expect_tx(&xw.full[i], stage_doubles * (uint32_t)sizeof(double));
            bulk_g2s(xw.ring + (size_t)i * stage_doubles, m.xT + ((size_t)(ks * 4 + warp) * m.ssd_nj) * 64, stage_doubles * (uint32_t)sizeof(double), &xw.full[i]);
        }
    }
    for (int ks = blockIdx.y * g.kpc; ks < ks_end; ++ks) {                 // (the operand ring carries over: xw.it_base)
        xw.ks = ks;
        const double *bsrc = bfrag + (((size_t)oct0 * m.n_ksplit + ks) * m.ssd_nj) * 32;
#define XD_CALL(NO, NJC, HF) xdot_body<NO, NJC, HF, STAGES>(m, bsrc, bstride, msrc, lv, ll_acc, oct0, T0, T1, xw, wait, tl, tlc, ahead ? 1 : 0)
        if (m.ssd_nj == SSD_NJ && m.ssd_half) {
            switch (noct) { case 4: if constexpr (MAXOCT >= 4) XD_CALL(4, SSD_NJ, true); break; case 3: if constexpr (MAXOCT >= 3) XD_CALL(3, SSD_NJ, true); break; case 2: XD_CALL(2, SSD_NJ, true); break; default: XD_CALL(1, SSD_NJ, true); break; }
        } else if (m.ssd_nj == SSD_NJ) {
            switch (noct) { case 4: if constexpr (MAXOCT >= 4) XD_CALL(4, SSD_NJ, false); break; case 3: if constexpr (MAXOCT >= 3) XD_CALL(3, SSD_NJ, false); break; case 2: XD_CALL(2, SSD_NJ, false); break; default: XD_CALL(1, SSD_NJ, false); break; }
        } else {
            switch (noct) { case 4: if constexpr (MAXOCT >= 4) XD_CALL(4, 0, false); break; case 3: if constexpr (MAXOCT >= 3) XD_CALL(3, 0, false); break; case 2: XD_CALL(2, 0, false); break; default: XD_CALL(1, 0, false); break; }
        }
#undef XD_CALL
    }
}

// centred means of arbitrary parameter vectors in the k_xdot layout (demcmc_eval, initial weights)
__global__ void __launch_bounds__(PA_THREADS) k_stage_means(ModelDev m, const double *theta, int64_t n, double *bfrag, double *magic,
                                                            long long *acc, double *q)
{
    const int64_t wi = ((int64_t)blockIdx.x * PA_THREADS + threadIdx.x) >> 5;
    if (wi >= n) return;
    stage_bfrag(m, theta + (size_t)wi * m.d, wi, bfrag, magic, acc + wi, q + wi, nullptr);
}

static int n_sms()
{
    static int sms[64] = { 0 };
    if (!sms[g_dev]) cudaDeviceGetAttribute(&sms[g_dev], cudaDevAttrMultiProcessorCount, g_dev);
    return sms[g_dev] > 0 ? sms[g_dev] : 148;
}

// A level's octets are dealt to particle tiles as evenly as possible (tiles of 3 and 4 octets rather
// than 4,4,..,1: a one-octet CTA has two DMMA chains and starves next to eight-chain warps), and
// the resident CTA slots of one wave are dealt to the tiles in proportion to their octets; a level
// too large for that is cut into many short CTAs instead.
static XdGrid xdot_grid(const ModelDev &m, int n, int slots, int max_oct, int max_kpc)
{
    XdGrid g;
    const int octets = (n + SSD_OCT - 1) / SSD_OCT;
    const int nt = (octets + max_oct - 1) / max_oct;
    g.oct_lo = octets / nt; g.oct_hi = g.oct_lo + 1;
    g.n_hi = octets - g.oct_lo * nt; g.n_lo = nt - g.n_hi;
    const int n_tiles = (int)(m.ssd_ld / SSD_TN);
    const int c_max = std::max(1, n_tiles / XD_MIN_TILES);
    const int per_split = std::max(1, slots / std::max(1, m.n_ksplit));
    if (2 * nt <= per_split) {                                     // one wave
        g.c_lo = std::min(c_max, std::max(1, per_split * g.oct_lo / octets));
        g.c_hi = g.n_hi ? std::min(c_max, std::max(1, per_split * g.oct_hi / octets)) : 1;
        // spend what the rounding left over on whichever class is slower
        for (;;) {
            const int left = per_split - (g.n_hi * g.c_hi + g.n_lo * g.c_lo);
            const bool hi_slower = g.n_hi && (int64_t)g.oct_hi * g.c_lo > (int64_t)g.oct_lo * g.c_hi;
            if (hi_slower && left >= g.n_hi && g.c_hi < c_max) ++g.c_hi;
            else if (left >= g.n_lo && g.c_lo < c_max) ++g.c_lo;
            else if (g.n_hi && left >= g.n_hi && g.c_hi < c_max) ++g.c_hi;
            else break;
        }
    } else {
        // several waves: many short CTAs, the hardware scheduler balances them as slots free up
        g.c_hi = g.c_lo = std::min(c_max, std::max(1, n_tiles / XD_WAVE_TILES));
    }
    g.kpc = 1;
    if (n_tiles <= XD_KPC_MAX_TILES && m.n_ksplit > 1) {
        static const int kpc_env = [] { const char *e = getenv("DEMCMC_XD_KPC"); return e ? atoi(e) : 0; }();     // A/B runs: 1 = off
        const int64_t ctas = (int64_t)(g.n_hi * g.c_hi + g.n_lo * g.c_lo) * m.n_ksplit;
        g.kpc = kpc_env > 0 ? std::min(kpc_env, (int)m.n_ksplit) : (int)std::min<int64_t>(m.n_ksplit, std::max<int64_t>(1, (ctas + slots - 1) / slots));
        g.kpc = std::min(g.kpc, max_kpc);
    }
    return g;
}

constexpr int XDS_STAGES = 2, XDS_MAXOCT = 2, XDS_CTAS_PER_SM = 4;      // the short-stream instantiation
static int launch_xdot(const ModelDev &m, const XdStage &xs, const Level &lv, long long *ll_acc)
{
    static bool attr_set[64] = { false };
    if (!attr_set[g_dev]) {
        CU(cudaFuncSetAttribute(k_xdot_t<XD_STAGES, 4, XD_CTAS_PER_SM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)xdot_smem_bytes(SSD_NJ)));
        CU(cudaFuncSetAttribute(k_xdot_t<XDS_STAGES, XDS_MAXOCT, XDS_CTAS_PER_SM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)xdot_smem_bytes(SSD_NJ, XDS_STAGES)));
        attr_set[g_dev] = true;
    }
    unsigned long long *tls = lv.ctxs ? tl_slot() : nullptr, *tlc = lv.ctxs ? tl_cta() : nullptr;
    static const bool short_on = [] { const char *e = getenv("DEMCMC_XD_SHORT"); return !(e && e[0] == '0'); }();       // A/B runs
    if (short_on && m.ssd_ld / SSD_TN <= XD_KPC_MAX_TILES && m.n_ksplit > 1) {
        const XdGrid g = xdot_grid(m, lv.n, XDS_CTAS_PER_SM * n_sms(), XDS_MAXOCT, XDS_STAGES);
        dim3 grid((unsigned)(g.n_hi * g.c_hi + g.n_lo * g.c_lo), (unsigned)((m.n_ksplit + g.kpc - 1) / g.kpc));
        CU(launch_chained(k_xdot_t<XDS_STAGES, XDS_MAXOCT, XDS_CTAS_PER_SM>, grid, dim3(XD_THREADS), xdot_smem_bytes(m.ssd_nj, XDS_STAGES), m, (const double *)xs.bfrag,
                          (const double *)xs.magic, lv, ll_acc, g, tls, tlc));
        LAUNCHED("k_xdot");
        return 0;
    }
    const XdGrid g = xdot_grid(m, lv.n, XD_CTAS_PER_SM * n_sms(), 4, XD_STAGES);
    dim3 grid((unsigned)(g.n_hi * g.c_hi + g.n_lo * g.c_lo), (unsigned)((m.n_ksplit + g.kpc - 1) / g.kpc));
    CU(launch_chained(k_xdot_t<XD_STAGES, 4, XD_CTAS_PER_SM>, grid, dim3(XD_THREADS), xdot_smem_bytes(m.ssd_nj), m, (const double *)xs.bfrag, (const double *)xs.magic, lv, ll_acc, g, tls, tlc));
    LAUNCHED("k_xdot");
    return 0;
}

// ------------------------------------------------------------------------------------------------
// The persistent chunk kernel: ALL levels of a chunk (up to 16 overlapped sweeps) in ONE launch,
// one CTA per SM, warp-specialised, no kernel boundary and no host involvement between levels.
//   warps 0-7   two "virtual CTAs" of k_xdot (4 warps each, same private TMA rings, same inner loop);
//               virtual CTA v walks the levels in order and takes the items (particle tile x
//               observation range x dimension split) v, v + 2*gridDim, ... of each
//   warps 8-9   scalar warps: one particle update at a time -- proposal (the body of k_propose) and,
//               once the update's likelihood has arrived, the Metropolis accept (the body of k_accept)
// Dependencies are counters in global memory (release on arrive, acquire on poll):
//   prop_done[tile]   proposals of a particle tile staged          -> its DMMA items may start
//   xdot_done[tile]   warps that have added their share to ll_acc  -> its accepts may start
//   acc_done[level]   accepts finished                             -> proposals of levels that depend on it
// Every level names the level its proposals wait for (`dep`): the previous level of the same lane.
// With two lanes (independent sets of groups) the levels of the lanes alternate, so the DMMA warps
// work on one lane while the scalar warps accept / propose the other: the tensor pipe never waits
// for the scalar part of the step.  The staging buffers of the means alternate between two copies
// (level parity), guarded by acc_done[level - 2].
// Deadlock freedom: every wait is on work that comes EARLIER in every warp's own program order
// (levels are walked in order by all warps; an accept waits for DMMA items of its own level, those
// wait for proposals of that level, those for accepts of earlier levels), and the launch is one CTA
// per SM, so all CTAs are resident.  A wait that lasts 20 s traps instead of hanging the device.
// ------------------------------------------------------------------------------------------------
constexpr int PK_MAX_LEVELS = 448;             // levels of all lanes of one chunk (kernel parameter block: 48 bytes each)
constexpr int PK_MAX_TILES = 8192;
constexpr int PK_WARPS = 16;                    // per CTA: 4 per SM sub-partition, 128 registers each at launch
constexpr int PK_THREADS = PK_WARPS * 32;
constexpr int PK_REGS_DMMA = 216, PK_REGS_HELPER = 56, PK_REGS_IDLE = 24;   // per sub-partition 2 * 216 + 56 + 24 = 512 = 4 * 128, the launch allocation
constexpr int PK_SCALAR_CTAS = 6;               // CTAs (SMs) given to the scalar warps: 96 warps, one update each per level of ~100 (7 / 8 CTAs, so that no warp has two
                                                // proposals in a level of 112: the proposal phase 16 -> 9 us, but 2.73 against 2.83 M updates/s -- the DMMA items deal worse over 141 SMs)

struct PLevel { int32_t order_off, n, n_items, dep, tile_base, pad; XdGrid g; };
struct PChunk {
    int32_t n_levels, lag, n_scalar_ctas, n_buf;      // n_buf: staging copies of the means (level l uses copy pl.pad = l % n_buf)
    const int32_t *order;
    const SweepCtx *ctxs;
    int32_t *acc_done, *prop_done, *xdot_done;       // zeroed before the launch
    double *bfrag[MAX_LANES], *magic[MAX_LANES];
    long long *ll_acc;
    unsigned long long *tl;                          // debug timeline [level][PT_WORDS] or nullptr
    PLevel lv[PK_MAX_LEVELS];
};

// particle tile of an octet / of a launch index, as k_xdot deals them (XdGrid)
__host__ __device__ __forceinline__ void xd_tile_of_octet(const XdGrid &g, int oct, int &tile, int &oct0, int &noct)
{
    const int nh = g.n_hi * g.oct_hi;
    if (oct < nh) { tile = oct / g.oct_hi; oct0 = tile * g.oct_hi; noct = g.oct_hi; }
    else { const int t = (oct - nh) / g.oct_lo; tile = g.n_hi + t; oct0 = nh + t * g.oct_lo; noct = g.oct_lo; }
}
__host__ __device__ __forceinline__ int xd_tile_ctas(const XdGrid &g, int tile) { return tile < g.n_hi ? g.c_hi : g.c_lo; }

__device__ __forceinline__ int ld_acquire(const int32_t *p)
{
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// every lane has fenced its own writes before lane 0 publishes
__device__ __forceinline__ void arrive(int32_t *ctr)
{
    // DEMCMC_ARRIVE_FENCE (compile-time A/B): the release below is cumulative over what lane 0 has observed, and the
    // other lanes' stores are ordered before it by the warp barrier; the explicit fence in front of it is belt and braces
#ifdef DEMCMC_ARRIVE_FENCE
    __threadfence();
#endif
    __syncwarp();
    if ((threadIdx.x & 31) == 0) asm volatile("red.release.gpu.global.add.s32 [%0], 1;\n" ::"l"(ctr) : "memory");
}

// the scalar warps are few (96) and sit on the critical path of a level: they poll without back-off
__device__ __forceinline__ void wait_ge_fast(const int32_t *ctr, int target)
{
    if (ld_acquire(ctr) >= target) return;
    const unsigned long long t0 = gtime();
    while (ld_acquire(ctr) < target) {
        __nanosleep(20);
        if (gtime() - t0 > 20000000000ull) __trap();
    }
}
struct FlagWait {
    const int32_t *c0; int t0; const int32_t *c1; int t1;
    unsigned long long *tl; int w_min, w_max;            // debug timeline: stamp when the wait is over
    mutable unsigned long long t_done;
    __device__ __forceinline__ void operator()() const
    {
        if (c0) wait_ge_fast(c0, t0);
        if (c1) wait_ge_fast(c1, t1);
        if (tl) {
            t_done = gtime();
            if ((threadIdx.x & 31) == 0) { if (w_min >= 0) atomicMax(tl + w_min, ~t_done); if (w_max >= 0) atomicMax(tl + w_max, t_done); }
        }
    }
};
// per level: stamps (min stored complemented) and, summed over the DMMA warps, the nanoseconds spent
// waiting for the proposals, in the item (B fragments, DMMA loop, flush) and in the arrive
enum { PT_P0 = 0, PT_PW, PT_P1, PT_XW0, PT_XW1, PT_X1, PT_AW0, PT_A1, PT_SUM_WAIT, PT_SUM_ITEM, PT_SUM_ARRIVE, PT_ITEMS,
       PT_S_PRE, PT_S_BODY, PT_S_STAGE, PT_S_ARR, PT_S_N, PT_A_BODY, PT_A_ARR, PT_A_N, PT_WORDS = 24 };
// (Tried and dropped: the DMMA warps deferring the arrive of a finished item behind the next item's
// B-fragment loads.  Carrying the pending counter across items made ptxas drop the raised register
// budget of the setmaxnreg region -- 125 registers, B fragments reloaded from local memory inside
// the DMMA loop.  The helper warps do that job now; scripts/regcheck.sh and
// tests/test_abi_library.py watch the register budget.)
struct FlagLanes : WarpLanes {
    FlagWait w;
    __device__ __forceinline__ void dependency_wait() const { w(); }
};
// a proposal whose dependency wait first runs the warp's own pending accepts: the state-independent
// prologue of the proposal (Philox plan, noise, bounds, prior specs) is then over before the
// likelihood of the level it waits for has even arrived
template <class PENDING>
struct ProposeLanes : WarpLanes {
    const PENDING &pending; FlagWait w;
    __device__ __forceinline__ ProposeLanes(const PENDING &p, const FlagWait &fw) : pending(p), w(fw) {}
    __device__ __forceinline__ void dependency_wait() const { pending(); w(); }
};

// one item of a level: (dimension split, particle tile, observation-tile range), as k_xdot's grid deals them
struct PkItem { int ks, tile, oct0, noct, T0, T1, n_in_tile; };
__device__ __forceinline__ PkItem pk_item(const PLevel &pl, int n_tiles, int q)
{
    PkItem it;
    const XdGrid &g = pl.g;
    it.ks = q / pl.n_items;
    const int bx = q - it.ks * pl.n_items;
    int c_in, C;
    const int n_in_hi = g.n_hi * g.c_hi;
    if (bx < n_in_hi) { it.tile = bx / g.c_hi; c_in = bx - it.tile * g.c_hi; C = g.c_hi; it.noct = g.oct_hi; it.oct0 = it.tile * g.oct_hi; }
    else { const int r = bx - n_in_hi, t = r / g.c_lo; it.tile = g.n_hi + t; c_in = r - t * g.c_lo; C = g.c_lo; it.noct = g.oct_lo; it.oct0 = g.n_hi * g.oct_hi + t * g.oct_lo; }
    it.T0 = (int)((int64_t)c_in * n_tiles / C); it.T1 = (int)((int64_t)(c_in + 1) * n_tiles / C);
    it.n_in_tile = min(pl.n, (it.oct0 + it.noct) * SSD_OCT) - it.oct0 * SSD_OCT;
    return it;
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}

// what the DMMA warps of a virtual CTA see of an item: the helper warp's shared-memory copy of the
// tile's B fragments (b_full), and the two signals back to it (b_empty: the copy is in registers;
// item_done: the cross terms are in ll_acc)
template <bool TL>
struct VctaHooks {
    uint64_t *b_full, *b_empty, *item_done;
    uint32_t parity;
    unsigned long long *tl; mutable unsigned long long t_done, t_first;   // debug timeline (TL) only
    __device__ __forceinline__ void operator()() const
    {
        mbar_wait(b_full, parity);
        if (TL && tl) {
            t_done = gtime();
            if ((threadIdx.x & 31) == 0) { atomicMax(tl + PT_XW0, ~t_done); atomicMax(tl + PT_XW1, t_done); }
        }
    }
    __device__ __forceinline__ void after_loads() const { if (TL && tl) t_first = gtime(); if ((threadIdx.x & 31) == 0) mbar_arrive(b_empty); }   // called right after a __syncwarp
    __device__ __forceinline__ void item_end() const { __syncwarp(); if ((threadIdx.x & 31) == 0) mbar_arrive(item_done); }
};

constexpr int PK_STAGES = 3;                    // ring depth of the persistent kernel (the fourth stage's memory holds the B copies)
static size_t pk_bbuf_doubles(int nj) { return (size_t)4 * nj * 32 + 4 * SSD_OCT; }
static size_t pk_smem_bytes(int nj)
{
    return sizeof(double) * ((size_t)8 * PK_STAGES * nj * 64 + 2 * pk_bbuf_doubles(nj)) + sizeof(uint64_t) * (8 * PK_STAGES + 6);
}

// TEMPER: as k_accept's (the untempered instantiations keep the registers, and the spills, they had before tempering)
template <bool TL, bool TEMPER>
__global__ void __launch_bounds__(PK_THREADS, 1) k_chunk_persist(const __grid_constant__ ConfigDev cfg, const __grid_constant__ ModelDev m,
                                                                 const __grid_constant__ PChunk ck)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // Roles.  The scalar part of the step (Philox, pow/log/exp, priors) runs on the same fp64 pipe as
    // DMMA: next to two DMMA warps a scalar warp's dependent fp64 chain takes 3-4x as long (measured:
    // 26 us instead of 8 per proposal).  So the last n_scalar_ctas CTAs are scalar-only (16 warps at
    // the launch's 128 registers).  In the DMMA CTAs warps 0-7 are the two virtual CTAs (setmaxnreg:
    // 216 registers each), warps 8 and 9 are their HELPERS (56 registers): a helper polls the
    // proposal counter of its virtual CTA's next item, copies that tile's B fragments and magic
    // constants into shared memory while the DMMA warps are still in the previous item, and
    // publishes a finished item (fence + xdot_done) on their behalf -- so the DMMA warps never touch
    // a global flag, never wait on an L2 round trip for their operands and never stall in a fence.
    // Warps 10-15 give their registers back and leave.
    const int n_dmma_ctas = (int)gridDim.x - ck.n_scalar_ctas;
    const bool scalar_cta = (int)blockIdx.x >= n_dmma_ctas;
    const int nj = m.ssd_nj;
    const uint32_t stage_doubles = (uint32_t)nj * 64;
    double *const ring0 = reinterpret_cast<double *>(smem_raw);
    double *const bbuf0 = ring0 + (size_t)8 * PK_STAGES * stage_doubles;
    const size_t bbuf_doubles = (size_t)4 * nj * 32 + 4 * SSD_OCT;
    uint64_t *const bars = reinterpret_cast<uint64_t *>(bbuf0 + 2 * bbuf_doubles);     // full[8][PK_STAGES], then per virtual CTA b_full, b_empty, item_done
    uint64_t *const vbars = bars + 8 * PK_STAGES;
    if (!scalar_cta) {
        if (threadIdx.x == 0) {
            for (int vc = 0; vc < 2; ++vc) { mbar_init(&vbars[vc * 3 + 0], 1); mbar_init(&vbars[vc * 3 + 1], 4); mbar_init(&vbars[vc * 3 + 2], 4); }
            asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
        }
        __syncthreads();                                         // the only CTA-wide barrier: before any warp leaves
    }
    const int n_tiles = (int)(m.ssd_ld / SSD_TN);
    if (!scalar_cta && warp >= 8) {
        if (warp >= 12) { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;\n" ::"n"(PK_REGS_IDLE)); return; }
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;\n" ::"n"(PK_REGS_HELPER));
        if (warp >= 10) return;
        // ---- helper warp of virtual CTA vc ----------------------------------------------------------
        const int vc = warp - 8, v = blockIdx.x * 2 + vc, NV = n_dmma_ctas * 2;
        double *const bbuf = bbuf0 + (size_t)vc * bbuf_doubles, *const mbuf = bbuf + (size_t)4 * nj * 32;
        uint64_t *const b_full = &vbars[vc * 3 + 0], *const b_empty = &vbars[vc * 3 + 1], *const item_done = &vbars[vc * 3 + 2];
        uint32_t n = 0;                                          // items handed to the DMMA warps so far
        int32_t *prev_ctr = nullptr;                             // xdot_done counter of the item they are working on
        auto publish = [&](int32_t *ctr) {
            __threadfence();
            __syncwarp();
            if (lane == 0) asm volatile("red.release.gpu.global.add.s32 [%0], 4;\n" ::"l"(ctr) : "memory");
        };
        for (int L = 0; L < ck.n_levels; ++L) {
            const PLevel &pl = ck.lv[L];
            const int total = pl.n_items * m.n_ksplit;
            for (int q = v; q < total; q += NV) {
                const PkItem it = pk_item(pl, n_tiles, q);
                int32_t *ctr = ck.xdot_done + pl.tile_base + it.tile;
                if (it.T1 <= it.T0) { publish(ctr); continue; }  // (k_xdot's grids never deal an empty range)
                const int32_t *flag = ck.prop_done + pl.tile_base + it.tile;
                const double *bsrc = ck.bfrag[pl.pad] + (((size_t)it.oct0 * m.n_ksplit + it.ks) * nj) * 32;
                const double *msrc = ck.magic[pl.pad] + (size_t)it.oct0 * SSD_OCT;
                const size_t bstride = (size_t)m.n_ksplit * nj * 32;
                bool filled = false;
                const unsigned long long t0 = gtime();
                while (prev_ctr || !filled) {
                    if (prev_ctr && mbar_try_wait(item_done, (n - 1) & 1u)) { publish(prev_ctr); prev_ctr = nullptr; }
                    if (!filled && (n == 0 || mbar_try_wait(b_empty, (n - 1) & 1u)) && ld_acquire(flag) >= it.n_in_tile) {
                        // the staged means were written with ordinary stores on other SMs and acquired just
                        // above; the copies read them through the async proxy, and complete on b_full
                        if (lane == 0) {
                            asm volatile("fence.proxy.async.global;\n" ::: "memory");
                            const uint32_t oct_bytes = (uint32_t)nj * 32 * sizeof(double), mg_bytes = (uint32_t)it.noct * SSD_OCT * sizeof(double);
                            mbar_expect_tx(b_full, oct_bytes * (uint32_t)it.noct + mg_bytes);
                            for (int pt = 0; pt < it.noct; ++pt) bulk_g2s(bbuf + (size_t)pt * nj * 32, bsrc + pt * bstride, oct_bytes, b_full);
                            bulk_g2s(mbuf, msrc, mg_bytes, b_full);
                        }
                        __syncwarp();
                        filled = true;
                    } else if (!filled || prev_ctr) {
                        __nanosleep(32);
                        if (gtime() - t0 > 20000000000ull) __trap();
                    }
                }
                prev_ctr = ctr; ++n;
            }
        }
        if (prev_ctr) { mbar_wait(item_done, (n - 1) & 1u); publish(prev_ctr); }
        return;
    }
    if (!scalar_cta) {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;\n" ::"n"(PK_REGS_DMMA));
        // ---- DMMA warps ---------------------------------------------------------------------------
        const int vc = warp >> 2, v = blockIdx.x * 2 + vc, NV = n_dmma_ctas * 2;
        XdWarp xw;
        xw.warp = warp & 3; xw.ks = 0; xw.it_base = 0;
        xw.ring = ring0 + (size_t)warp * PK_STAGES * stage_doubles;
        xw.full = bars + warp * PK_STAGES;
        if (lane == 0) {
#pragma unroll
            for (int s = 0; s < PK_STAGES; ++s) mbar_init(&xw.full[s], 1);
            asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
        }
        __syncwarp();
        const double *const bbuf = bbuf0 + (size_t)vc * bbuf_doubles, *const mbuf = bbuf + (size_t)4 * nj * 32;
        uint32_t n = 0;
        for (int L = 0; L < ck.n_levels; ++L) {
            const PLevel &pl = ck.lv[L];
            Level lv; lv.order = ck.order + pl.order_off; lv.n = pl.n; lv.ctxs = ck.ctxs;
            const int total = pl.n_items * m.n_ksplit;
            for (int q = v; q < total; q += NV) {
                const PkItem it = pk_item(pl, n_tiles, q);
                if (it.T1 <= it.T0) continue;
                unsigned long long *tl = (TL && ck.tl) ? ck.tl + (size_t)L * PT_WORDS : nullptr;
                const VctaHooks<TL> hooks = { &vbars[vc * 3 + 0], &vbars[vc * 3 + 1], &vbars[vc * 3 + 2], n & 1u, tl, 0ull, 0ull };
                const unsigned long long t_a = (TL && tl) ? gtime() : 0ull;
                xw.ks = it.ks;
                const int oct0 = it.oct0, T0 = it.T0, T1 = it.T1;
                const size_t bstride = (size_t)nj * 32;
#define PK_CALL(NO, NJC, HF) xdot_body<NO, NJC, HF, PK_STAGES>(m, bbuf, bstride, mbuf, lv, ck.ll_acc, oct0, T0, T1, xw, hooks, nullptr, nullptr)
                if (m.ssd_nj == SSD_NJ && m.ssd_half) {
                    switch (it.noct) { case 4: PK_CALL(4, SSD_NJ, true); break; case 3: PK_CALL(3, SSD_NJ, true); break; case 2: PK_CALL(2, SSD_NJ, true); break; default: PK_CALL(1, SSD_NJ, true); break; }
                } else if (m.ssd_nj == SSD_NJ) {
                    switch (it.noct) { case 4: PK_CALL(4, SSD_NJ, false); break; case 3: PK_CALL(3, SSD_NJ, false); break; case 2: PK_CALL(2, SSD_NJ, false); break; default: PK_CALL(1, SSD_NJ, false); break; }
                } else {
                    switch (it.noct) { case 4: PK_CALL(4, 0, false); break; case 3: PK_CALL(3, 0, false); break; case 2: PK_CALL(2, 0, false); break; default: PK_CALL(1, 0, false); break; }
                }
#undef PK_CALL
                ++n;
                if (TL && tl && lane == 0) {
                    const unsigned long long t_b = gtime();
                    atomicMax(tl + PT_X1, t_b);
                    atomicAdd(tl + PT_SUM_WAIT, hooks.t_done - t_a); atomicAdd(tl + PT_SUM_ITEM, t_b - hooks.t_done);
                    atomicAdd(tl + PT_SUM_ARRIVE, hooks.t_first - hooks.t_done);      // B fragments + first observation tile (of T1 - T0)
                    atomicAdd(tl + PT_ITEMS, 1ull);
                }
            }
        }
        return;
    }
    // ---- scalar warps ---------------------------------------------------------------------------
    const int sw = ((int)blockIdx.x - n_dmma_ctas) * PK_WARPS + warp, NS = ck.n_scalar_ctas * PK_WARPS;
    auto accept_level = [&](int L) {
        const PLevel &pl = ck.lv[L];
        for (int wi = sw; wi < pl.n; wi += NS) {
            const uint32_t e = (uint32_t)ck.order[pl.order_off + wi];
            const SweepCtx ctx = ck.ctxs[e >> LV_SLOT_SHIFT];
            int tile, oct0, noct;
            xd_tile_of_octet(pl.g, wi / SSD_OCT, tile, oct0, noct);
            FlagLanes co;
            unsigned long long *tl = (TL && ck.tl) ? ck.tl + (size_t)L * PT_WORDS : nullptr;
            co.w = { ck.xdot_done + pl.tile_base + tile, xd_tile_ctas(pl.g, tile) * 4 * m.n_ksplit, nullptr, 0, tl, PT_AW0, -1, 0ull };
            accept_particle<FlagLanes, TEMPER>(co, cfg, m, ctx, (int)(e & LV_POS_MASK));
            const unsigned long long ta1 = (TL && tl) ? gtime() : 0ull;
            arrive(ck.acc_done + L);
            if (TL && tl && lane == 0) {
                const unsigned long long ta2 = gtime();
                atomicMax(tl + PT_A1, ta2);
                atomicAdd(tl + PT_A_BODY, ta1 - co.w.t_done); atomicAdd(tl + PT_A_ARR, ta2 - ta1); atomicAdd(tl + PT_A_N, 1ull);
            }
        }
    };
    int next_acc = 0;
    for (int L = 0; L < ck.n_levels; ++L) {
        const PLevel &pl = ck.lv[L];
        // the accepts this level's proposals (or its staging buffer) wait for: inside the first
        // proposal's dependency wait when this warp has one, else here
        const int must = max(pl.dep, L - ck.n_buf);
        auto pending = [&]() { while (next_acc <= must) accept_level(next_acc++); };
        for (int wi = sw; wi < pl.n; wi += NS) {
            const uint32_t e = (uint32_t)ck.order[pl.order_off + wi];
            const SweepCtx ctx = ck.ctxs[e >> LV_SLOT_SHIFT];
            const int p = (int)(e & LV_POS_MASK);
            double *bfrag = ck.bfrag[pl.pad], *magic = ck.magic[pl.pad];
            unsigned long long *tl = (TL && ck.tl) ? ck.tl + (size_t)L * PT_WORDS : nullptr;
            const unsigned long long tp0 = (TL && tl) ? gtime() : 0ull;
            if (tl && lane == 0) atomicMax(tl + PT_P0, ~tp0);
            const FlagWait fw = { pl.dep >= 0 ? ck.acc_done + pl.dep : nullptr, pl.dep >= 0 ? ck.lv[pl.dep].n : 0,
                                  L >= ck.n_buf ? ck.acc_done + (L - ck.n_buf) : nullptr, L >= ck.n_buf ? ck.lv[L - ck.n_buf].n : 0, tl, PT_PW, -1, 0ull };
            const ProposeLanes<decltype(pending)> co(pending, fw);
            StageSink sink = { m, bfrag, wi, m.kind == M_MVNORMAL, { 0.0 }, 0.0 };
            propose_particle(co, cfg, m, ctx, p, sink);
            const unsigned long long tp1 = (TL && tl) ? gtime() : 0ull;
            if (sink.on) stage_scale(m, warp_sum(sink.msq), wi, magic, ctx.ll_acc + p, ctx.ll_q + p, ctx.prop_msq + p);
            else {
                __syncwarp();
                stage_bfrag(m, ctx.prop_theta + (size_t)p * cfg.d, wi, bfrag, magic, ctx.ll_acc + p, ctx.ll_q + p, ctx.prop_msq + p);
            }
            int tile, oct0, noct;
            xd_tile_of_octet(pl.g, wi / SSD_OCT, tile, oct0, noct);
            const unsigned long long tp2 = (TL && tl) ? gtime() : 0ull;
            arrive(ck.prop_done + pl.tile_base + tile);
            if (TL && tl && lane == 0) {
                const unsigned long long tp3 = gtime();
                atomicMax(tl + PT_P1, tp3);
                // prologue + pending accepts + dependency wait | body | staging | arrive
                atomicAdd(tl + PT_S_PRE, co.w.t_done - tp0); atomicAdd(tl + PT_S_BODY, tp1 - co.w.t_done);
                atomicAdd(tl + PT_S_STAGE, tp2 - tp1); atomicAdd(tl + PT_S_ARR, tp3 - tp2); atomicAdd(tl + PT_S_N, 1ull);
            }
        }
        pending();                                           // a warp without a proposal in this level
        if (ck.lag == 0) while (next_acc <= L) accept_level(next_acc++);
    }
    while (next_acc < ck.n_levels) accept_level(next_acc++);
}

static XdGrid xdot_grid(const ModelDev &m, int n, int slots, int max_oct = 4, int max_kpc = XD_STAGES);

// debug timeline of the persistent kernel (DEMCMC_PK_TIMELINE=<levels> DEMCMC_PK_TIMELINE_FILE=<csv>)
static unsigned long long *g_ptl = nullptr;
static int g_ptl_cap = -1, g_ptl_level = 0;
static std::vector<int> g_ptl_n, g_ptl_chunk;
static void pk_timeline_dump()
{
    const char *path = getenv("DEMCMC_PK_TIMELINE_FILE");
    if (g_ptl_cap <= 0 || !g_ptl || !path || g_ptl_level == 0) return;
    cudaDeviceSynchronize();
    const int n = g_ptl_level;
    std::vector<unsigned long long> h((size_t)PT_WORDS * n);
    if (cudaMemcpy(h.data(), g_ptl, sizeof(unsigned long long) * h.size(), cudaMemcpyDeviceToHost) != cudaSuccess) return;
    FILE *f = fopen(path, "w");
    if (!f) return;
    fprintf(f, "level,chunk,n,propose_first_start,propose_dep_ready,propose_last_end,xdot_first_ready,xdot_last_ready,xdot_last_end,accept_first_ready,accept_last_end,warp_items,wait_us_per_item,work_us_per_item,arrive_us_per_item,prop_pre_us,prop_body_us,prop_stage_us,prop_arrive_us,acc_body_us,acc_arrive_us\n");
    unsigned long long t0 = ~0ull;
    for (int i = 0; i < n; ++i) if (h[(size_t)i * PT_WORDS + PT_P0]) t0 = std::min(t0, ~h[(size_t)i * PT_WORDS + PT_P0]);
    auto rel = [&](unsigned long long v) { return v ? (double)((long long)(v - t0)) * 1e-3 : -1.0; };
    for (int i = 0; i < n; ++i) {
        const unsigned long long *w = h.data() + (size_t)i * PT_WORDS;
        const double ni = w[PT_ITEMS] ? (double)w[PT_ITEMS] : 1.0;
        const double ns = w[PT_S_N] ? (double)w[PT_S_N] * 1e3 : 1.0, na = w[PT_A_N] ? (double)w[PT_A_N] * 1e3 : 1.0;
        fprintf(f, "%d,%d,%d,%.3f,%.3f,%.3f,%.3f,%.3f,%.3f,%.3f,%.3f,%llu,%.3f,%.3f,%.3f,%.3f,%.3f,%.3f,%.3f,%.3f,%.3f\n", i, g_ptl_chunk[i], g_ptl_n[i], rel(~w[PT_P0]), rel(~w[PT_PW]), rel(w[PT_P1]),
                rel(~w[PT_XW0]), rel(w[PT_XW1]), rel(w[PT_X1]), rel(~w[PT_AW0]), rel(w[PT_A1]), w[PT_ITEMS],
                (double)w[PT_SUM_WAIT] * 1e-3 / ni, (double)w[PT_SUM_ITEM] * 1e-3 / ni, (double)w[PT_SUM_ARRIVE] * 1e-3 / ni,
                (double)w[PT_S_PRE] / ns, (double)w[PT_S_BODY] / ns, (double)w[PT_S_STAGE] / ns, (double)w[PT_S_ARR] / ns,
                (double)w[PT_A_BODY] / na, (double)w[PT_A_ARR] / na);
    }
    fclose(f);
}

static int persist_enabled()                                  // DEMCMC_PERSIST=0: level-by-level launches (A/B runs, tests)
{
    const char *e = getenv("DEMCMC_PERSIST");
    return (e && e[0] == '0') ? 0 : 1;
}
static int persist_scalar_ctas()
{
    static int n_scalar = -1;
    if (n_scalar < 0) { const char *e = getenv("DEMCMC_PK_SCALAR_CTAS"); n_scalar = e ? std::max(1, std::min(atoi(e), 64)) : PK_SCALAR_CTAS; }
    return n_scalar;
}
// How many lanes (independent sets of groups with alternating levels) the persistent kernel wants
// for this job, or 0 when the job is better served level by level: other models, a single group
// (nothing to alternate with: the scalar part of every level would sit on the critical path with
// fewer warps than k_propose has), or levels far larger than the scalar warps.
int chunk_persist_lanes(const ConfigDev &cfg, const ModelDev &m)
{
    if (!persist_enabled() || !is_ssd(m.kind)) return 0;
    if (cfg.G_local < 2) return 0;
    if ((int64_t)cfg.G_local * cfg.Np / 8 > (int64_t)4 * PK_WARPS * persist_scalar_ctas()) return 0;   // ~ a level per lane
    // Two lanes.  More (DEMCMC_PK_LANES = 3, 4: one lane per group) give a lane's accept -> propose chain more DMMA time
    // to hide in, but halve the levels: measured on configs[1] 2 / 3 / 4 lanes = 2.76 / 2.65 / 2.52 M updates/s -- smaller
    // particle tiles (fewer octets per streamed A fragment) and twice the items cost more than the waits they remove.
    static int want = -1;
    if (want < 0) { const char *e = getenv("DEMCMC_PK_LANES"); want = e ? std::max(2, std::min(atoi(e), (int)MAX_LANES)) : 2; }
    return std::min(cfg.G_local, want);
}

// Runs the levels [level_off[l], level_off[l] + level_n[l]) of a chunk (entries in d_order) in one persistent
// launch.  dep[l] = the level whose accepts the proposals of level l wait for (-1: none), lag = how
// many levels the accepts trail the proposals in the scalar warps' program (0 or 1).
// Returns 1 when the chunk does not fit this kernel (the caller launches the levels one by one).
int launch_chunk_persist(const ConfigDev &cfg, const ModelDev &m, const int32_t *d_order, const SweepCtx *d_ctx,
                         const int32_t *level_off, const int32_t *level_n, const int32_t *dep, int n_levels, int lag, long long *ll_acc, int n_buf)
{
    n_buf = std::max(2, std::min(n_buf, (int)MAX_LANES));
    if (!persist_enabled() || !is_ssd(m.kind) || n_levels <= 0 || n_levels > PK_MAX_LEVELS) return 1;
    static thread_local PChunk ck;                           // 9 KB: not on the stack of every call
    const int n_scalar = persist_scalar_ctas();
    const int sms = n_sms(), slots = XD_CTAS_PER_SM * (sms - n_scalar);
    int tiles = 0, n_max = 0;
    for (int l = 0; l < n_levels; ++l) {
        PLevel &pl = ck.lv[l];
        pl.order_off = level_off[l]; pl.n = level_n[l]; pl.dep = dep[l]; pl.tile_base = tiles; pl.pad = l % n_buf;
        if (pl.n <= 0 || pl.dep >= l) return 1;
        pl.g = xdot_grid(m, pl.n, slots);
        pl.n_items = pl.g.n_hi * pl.g.c_hi + pl.g.n_lo * pl.g.c_lo;
        tiles += pl.g.n_hi + pl.g.n_lo;
        n_max = std::max(n_max, pl.n);
    }
    if (tiles > PK_MAX_TILES) return 1;
    // the scalar warps take one update at a time: levels far larger than their number are better
    // served by the wide propose / accept kernels of the level-by-level path
    if (n_max > 8 * PK_WARPS * n_scalar) return 1;
    static int32_t *ctr[64] = { nullptr };
    if (!ctr[g_dev]) CU(cudaMalloc(&ctr[g_dev], sizeof(int32_t) * (PK_MAX_LEVELS + 2 * PK_MAX_TILES)));
    XdStage *xs[MAX_LANES];
    const int keep = g_lane;
    for (int b = 0; b < n_buf; ++b) {
        g_lane = b;
        xs[b] = xd_stage(m, std::max(n_max, cfg.G_local * cfg.Np));
        if (!xs[b]) { g_lane = keep; return -1; }
        // the copy was cleared on lane b's stream; this kernel runs on the launching lane's: order them
        if (xs[b]->fresh && b != keep) { cudaStreamSynchronize(stream()); }
        xs[b]->fresh = false;
    }
    g_lane = keep;
    ck.n_levels = n_levels; ck.lag = lag; ck.n_scalar_ctas = n_scalar; ck.n_buf = n_buf; ck.order = d_order; ck.ctxs = d_ctx;
    ck.acc_done = ctr[g_dev]; ck.prop_done = ctr[g_dev] + PK_MAX_LEVELS; ck.xdot_done = ck.prop_done + PK_MAX_TILES;
    for (int b = 0; b < n_buf; ++b) { ck.bfrag[b] = xs[b]->bfrag; ck.magic[b] = xs[b]->magic; }
    ck.ll_acc = ll_acc;
    if (g_ptl_cap < 0) {
        const char *e = getenv("DEMCMC_PK_TIMELINE");
        g_ptl_cap = e ? atoi(e) : 0;
        if (g_ptl_cap > 0 && (cudaMalloc(&g_ptl, sizeof(unsigned long long) * PT_WORDS * g_ptl_cap) != cudaSuccess ||
                              cudaMemset(g_ptl, 0, sizeof(unsigned long long) * PT_WORDS * g_ptl_cap) != cudaSuccess)) g_ptl_cap = 0;
    }
    ck.tl = nullptr;
    if (g_ptl_cap > 0 && g_ptl_level + n_levels <= g_ptl_cap) {
        static int chunk_no = 0;
        ck.tl = g_ptl + (size_t)PT_WORDS * g_ptl_level;
        for (int l = 0; l < n_levels; ++l) { g_ptl_n.push_back(ck.lv[l].n); g_ptl_chunk.push_back(chunk_no); }
        g_ptl_level += n_levels; ++chunk_no;
    }
    CU(cudaMemsetAsync(ctr[g_dev], 0, sizeof(int32_t) * (PK_MAX_LEVELS + PK_MAX_TILES + (size_t)tiles), stream()));
    static bool attr_set[64] = { false };
    const size_t smem = pk_smem_bytes(m.ssd_nj);
    if (!attr_set[g_dev]) {
        CU(cudaFuncSetAttribute(k_chunk_persist<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pk_smem_bytes(SSD_NJ)));
        CU(cudaFuncSetAttribute(k_chunk_persist<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pk_smem_bytes(SSD_NJ)));
        CU(cudaFuncSetAttribute(k_chunk_persist<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pk_smem_bytes(SSD_NJ)));
        CU(cudaFuncSetAttribute(k_chunk_persist<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pk_smem_bytes(SSD_NJ)));
        attr_set[g_dev] = true;
    }
    // a cooperative launch: CUDA itself guarantees (or refuses) that all CTAs are resident at once,
    // which is what the counter waits between CTAs rely on
    cudaLaunchConfig_t lc = {};
    lc.gridDim = dim3(sms); lc.blockDim = dim3(PK_THREADS); lc.dynamicSmemBytes = smem; lc.stream = stream();
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeCooperative;
    at[0].val.cooperative = 1;
    lc.attrs = at; lc.numAttrs = 1;
    const cudaError_t le = cfg.temp ? (ck.tl ? cudaLaunchKernelEx(&lc, k_chunk_persist<true, true>, cfg, m, ck) : cudaLaunchKernelEx(&lc, k_chunk_persist<false, true>, cfg, m, ck))
                                    : (ck.tl ? cudaLaunchKernelEx(&lc, k_chunk_persist<true, false>, cfg, m, ck) : cudaLaunchKernelEx(&lc, k_chunk_persist<false, false>, cfg, m, ck));
    if (le == cudaErrorCooperativeLaunchTooLarge) { (void)cudaGetLastError(); return 1; }   // not all resident here: level by level
    if (le != cudaSuccess) return cu_fail(le, "k_chunk_persist");
    LAUNCHED("k_chunk_persist");
    return 0;
}

// ------------------------------------------------------------------------------------------------
// user-written likelihoods (M_CUSTOM): the caller's per-observation density (include/demcmc_b200.h: DEMCMC_CUSTOM) is
// compiled at run time with NVRTC into k_ll_custom, the structure of k_ll_pointwise<M_GAUSSIAN> specialised to that
// density: PW_TP particles x one observation split per CTA, the same split partition, the same summation order
// (thread-strided, warp shuffle, CTA in warp order), and the same ll_part slots, which accept_particle / k_eval_finish
// reduce as for the registered pointwise kinds.  libnvrtc is loaded with dlopen, so the library still loads (and every
// registered kind still runs) where it is missing.  The kernel is plain-launched (no programmatic dependent launch):
// k_propose triggers its dependents early and k_ll_custom has no griddepcontrol.wait before it reads the proposals.
// ------------------------------------------------------------------------------------------------
static_assert(PW_TP == 8 && PW_THREADS == 256 && LV_POS_MASK == 0xFFFFFFu, "k_ll_custom's source spells these out");

// ahead of the user's text: calls of demcmc_obs / demcmc_particle that the source does not define resolve to these
// stand-ins (a definition in the source matches `const double *` exactly, these need a user-defined conversion); they
// add 0, and their return type tells the kernel source which of the two the user wrote
static const char CUSTOM_PRELUDE[] = R"CU(
#define DEMCMC_INF __longlong_as_double(0x7ff0000000000000LL)
#define DEMCMC_NAN __longlong_as_double(0x7ff8000000000000LL)
struct demcmc_zero_ { __device__ operator double() const { return 0.0; } };
struct demcmc_any_ptr_ { __device__ demcmc_any_ptr_(const double *) {} };
__device__ inline demcmc_zero_ demcmc_obs(demcmc_any_ptr_, demcmc_any_ptr_) { return demcmc_zero_(); }
__device__ inline demcmc_zero_ demcmc_particle(demcmc_any_ptr_) { return demcmc_zero_(); }
#line 1 "user.cu"
)CU";

// after it: the likelihood kernel (k_ll_pointwise's Gaussian form with the density inlined)
static const char CUSTOM_KERNEL[] = R"CU(
#line 1 "demcmc_custom_kernel.cu"
template <class T> struct demcmc_is_double_ { enum { value = 0 }; };
template <> struct demcmc_is_double_<double> { enum { value = 1 }; };
constexpr int demcmc_has_obs_ = demcmc_is_double_<decltype(demcmc_obs((const double *)0, (const double *)0))>::value;
constexpr int demcmc_has_particle_ = demcmc_is_double_<decltype(demcmc_particle((const double *)0))>::value;
static_assert(demcmc_has_obs_ || demcmc_has_particle_, "the source must define  __device__ double demcmc_obs(const double *par, "
              "const double *x)  (or, for a likelihood without observations, __device__ double demcmc_particle(const double *theta))");
// read by the host when the module is loaded: a model with observations needs demcmc_obs
extern "C" __device__ int demcmc_custom_has_obs = demcmc_has_obs_;
#ifdef DEMCMC_NPAR
static_assert(DEMCMC_NPAR >= 1, "DEMCMC_NPAR must be at least 1");
static_assert(DEMCMC_NPAR <= 256, "DEMCMC_NPAR is above DEMCMC_CUSTOM_MAX_PAR (256)");
#define DEMCMC_PAR_LEN_ (DEMCMC_NPAR)
#else
#define DEMCMC_PAR_LEN_ 256
#endif

extern "C" __global__ void __launch_bounds__(256) k_ll_custom(const double *theta, int d, const int *order, int n, const double *x,
                                                              int n_cols, long long n_obs, int split_len, int n_split, double *part)
{
    __shared__ double par[8][DEMCMC_PAR_LEN_];
    __shared__ double red[8][8];
    const int tile = blockIdx.x, split = blockIdx.y, tid = threadIdx.x;
    const int nt = min(8, n - tile * 8);
#ifdef DEMCMC_NPAR
    if (tid < nt) {
        const int p = order ? (int)((unsigned)order[tile * 8 + tid] & 0xFFFFFFu) : tile * 8 + tid;
        demcmc_prepare(theta + (size_t)p * d, par[tid]);
    }
#else
    for (int e = tid; e < nt * d; e += 256) {
        const int t = e / d, k = e - t * d;
        const int p = order ? (int)((unsigned)order[tile * 8 + t] & 0xFFFFFFu) : tile * 8 + t;
        par[t][k] = theta[(size_t)p * d + k];
    }
#endif
    __syncthreads();
    double acc[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) acc[t] = 0.0;
    const long long i0 = (long long)split * split_len;
    const long long i1 = min(n_obs, i0 + (long long)split_len);
    for (long long i = i0 + tid; i < i1; i += 256) {
        const double *xi = x + (size_t)i * n_cols;
#pragma unroll
        for (int t = 0; t < 8; ++t)
            if (t < nt) acc[t] += (double)demcmc_obs(par[t], xi);
    }
#pragma unroll
    for (int t = 0; t < 8; ++t) {
        double v = acc[t];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((tid & 31) == 0) red[tid >> 5][t] = v;
    }
    __syncthreads();
    if (tid < nt) {
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) v += red[w][tid];
        const int p = order ? (int)((unsigned)order[tile * 8 + tid] & 0xFFFFFFu) : tile * 8 + tid;
        if (demcmc_has_particle_ && split == 0) v += (double)demcmc_particle(theta + (size_t)p * d);
        part[(size_t)p * n_split + split] = v;
    }
}

// demcmc_eval_pointwise / demcmc_loo: every demcmc_obs value of 32 draws (one per lane) x 64 observations (8 per warp),
// written to out[obs][draw] instead of summed (kernels.cu: k_ll_obs).  Each draw's par row sits in dynamic shared memory,
// its length made odd so that the lanes' rows start in different banks; the host reads the length from demcmc_custom_npar.
#ifdef DEMCMC_NPAR
extern "C" __device__ int demcmc_custom_npar = DEMCMC_NPAR;
#else
extern "C" __device__ int demcmc_custom_npar = 0;
#endif
extern "C" __global__ void __launch_bounds__(256) k_ll_custom_obs(const double *theta, int d, long long n, const double *x, int n_cols,
                                                                  long long obs0, long long n_obs, double *out)
{
    extern __shared__ double demcmc_pars_[];
#ifdef DEMCMC_NPAR
    const int row = DEMCMC_NPAR | 1;
#else
    const int row = d | 1;
#endif
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long s0 = (long long)blockIdx.y * 32, i0 = (long long)blockIdx.x * 64;
#ifdef DEMCMC_NPAR
    if (threadIdx.x < 32 && s0 + threadIdx.x < n) demcmc_prepare(theta + (size_t)(s0 + threadIdx.x) * d, demcmc_pars_ + threadIdx.x * row);
#else
    for (int e = threadIdx.x; e < 32 * d; e += 256) {
        const int t = e / d, k = e - t * d;
        if (s0 + t < n) demcmc_pars_[t * row + k] = theta[(size_t)(s0 + t) * d + k];
    }
#endif
    __syncthreads();
    if (s0 + lane >= n) return;
    const double *par = demcmc_pars_ + lane * row;
    const int no = (int)min(64LL, n_obs - i0);
    for (int o = warp; o < no; o += 8)
        out[(size_t)(i0 + o) * n + s0 + lane] = (double)demcmc_obs(par, x + (size_t)(obs0 + i0 + o) * n_cols);
}
)CU";

// ------------------------------------------------------------------------------------------------
// simulation-based likelihoods (M_SIMULATED): the caller's simulator (include/demcmc_b200.h: DEMCMC_SIMULATED) is compiled
// at run time into two kernels around it, k_ll_sim (a level's proposals, writing the ll_part slots k_ll_custom writes, so
// accept, k_eval_finish and finalize_ll are unchanged) and k_ll_sim_obs (out[obs][draw] for launch_pointwise).  A CTA takes
// one parameter vector and one range of observations: it regenerates that vector's M simulations from their counter-based
// streams into shared memory (no global staging, no inter-CTA sync), sorts them by (label, value) with k_psis's
// order-preserving keys and bitonic network (spelled out again here: the run-time module cannot link the library's device
// code), takes each label's moments and quartiles, and streams its observations against their own label's group, one
// observation per warp.  Both kernels call the same two functions with the same 256 threads, so an observation's value is
// the same bits in either.  Plain launches (no programmatic dependent launch), like k_ll_custom.  The README's LBA
// simulator (DEMCMC_NPAR 5) compiled by libnvrtc 12.9 with this file's options plus --ptxas-options=-v: both kernels 64
// registers, no spills, 320 bytes of static shared memory (2336 without DEMCMC_NPAR: par[] is then 256 doubles); k_ll_sim
// has a 16-byte stack frame (y[2], passed to demcmc_simulate).  Dynamic shared memory: 9 bytes per simulation, padded to a
// power of two (144 KB at M = 16384).  The inner loop of demcmc_sim_obs_ issues 24 fp64 instructions per term (16 DFMA,
// 4 DMUL, 3 DADD, 1 DSETP; unrolled by 8 in the SASS).
// ------------------------------------------------------------------------------------------------
static_assert(offsetof(SweepCtx, sweep) == 0, "k_ll_sim reads a level's sweep as the first word of its SweepCtx");
static_assert(SIM_MAX_LABELS == 8 && SIM_SWEEP_EVAL == 0xFFFFFFFFu, "k_ll_sim's source spells these out");

// dynamic shared memory of k_ll_sim / k_ll_sim_obs: a key and a label per simulation, padded to a power of two (>= 16)
static size_t sim_smem(int M) { int p = 16; while (p < M) p <<= 1; return (size_t)p * (sizeof(unsigned long long) + 1); }

// ahead of the user's text: the random streams, and a stand-in demcmc_simulate whose return type tells the kernel source
// that the user wrote none (a definition in the source matches the argument types exactly, the stand-in needs conversions)
static const char SIM_PRELUDE[] = R"CU(
#define DEMCMC_INF __longlong_as_double(0x7ff0000000000000LL)
#define DEMCMC_NAN __longlong_as_double(0x7ff8000000000000LL)
struct demcmc_rng { unsigned c, unit, sweep, stream, k0, k1; int has_u, has_z; double u, z; };
struct demcmc_u4_ { unsigned x, y, z, w; };
__device__ inline demcmc_u4_ demcmc_philox_(demcmc_u4_ c, unsigned k0, unsigned k1)
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const unsigned hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const unsigned hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        demcmc_u4_ n;
        n.x = hi1 ^ c.y ^ k0; n.y = lo1; n.z = hi0 ^ c.w ^ k1; n.w = lo0;
        c = n;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return c;
}
__device__ inline double demcmc_u53_(unsigned lo, unsigned hi)
{
    const unsigned long long b = (((unsigned long long)hi << 32) | lo) >> 11;
    return b ? (double)b * 0x1.0p-53 : 0x1.0p-54;
}
__device__ inline double demcmc_uniform(demcmc_rng *r)
{
    if (r->has_u) { r->has_u = 0; return r->u; }
    demcmc_u4_ c; c.x = r->c++; c.y = r->unit; c.z = r->sweep; c.w = r->stream;
    const demcmc_u4_ o = demcmc_philox_(c, r->k0, r->k1);
    r->u = demcmc_u53_(o.z, o.w); r->has_u = 1;
    return demcmc_u53_(o.x, o.y);
}
__device__ inline double demcmc_normal(demcmc_rng *r)
{
    if (r->has_z) { r->has_z = 0; return r->z; }
    const double u1 = demcmc_uniform(r), u2 = demcmc_uniform(r);
    const double rad = sqrt(-2.0 * log(u1));
    double s, c;
    sincospi(2.0 * u2, &s, &c);
    r->z = rad * s; r->has_z = 1;
    return rad * c;
}
struct demcmc_missing_ {};
struct demcmc_any_cptr_ { __device__ demcmc_any_cptr_(const double *) {} };
struct demcmc_any_rng_ { __device__ demcmc_any_rng_(demcmc_rng *) {} };
struct demcmc_any_ptr_ { __device__ demcmc_any_ptr_(double *) {} };
__device__ inline demcmc_missing_ demcmc_simulate(demcmc_any_cptr_, demcmc_any_rng_, demcmc_any_ptr_) { return demcmc_missing_(); }
#line 1 "user.cu"
)CU";

static const char SIM_KERNEL[] = R"CU(
#line 1 "demcmc_sim_kernel.cu"
template <class T> struct demcmc_is_void_ { enum { value = 0 }; };
template <> struct demcmc_is_void_<void> { enum { value = 1 }; };
static_assert(demcmc_is_void_<decltype(demcmc_simulate((const double *)0, (demcmc_rng *)0, (double *)0))>::value,
              "the source must define  __device__ void demcmc_simulate(const double *par, demcmc_rng *rng, double *y)");
#ifdef DEMCMC_NPAR
static_assert(DEMCMC_NPAR >= 1, "DEMCMC_NPAR must be at least 1");
static_assert(DEMCMC_NPAR <= 256, "DEMCMC_NPAR is above DEMCMC_CUSTOM_MAX_PAR (256)");
#define DEMCMC_PAR_LEN_ (DEMCMC_NPAR)
#else
#define DEMCMC_PAR_LEN_ 256
#endif

// exp(x) for x <= 0 (de_math.h: de_exp_nonpos, the LBA kernel's): 2^k Taylor_13(r), |r| <= ln2 / 2; 0 below -708
__constant__ double demcmc_exp_c_[14] = {
    1.0, 1.0, 0.5, 1.0 / 6.0, 1.0 / 24.0, 1.0 / 120.0, 1.0 / 720.0, 1.0 / 5040.0, 1.0 / 40320.0, 1.0 / 362880.0, 1.0 / 3628800.0,
    1.0 / 39916800.0, 1.0 / 479001600.0, 1.0 / 6227020800.0
};
__device__ __forceinline__ double demcmc_exp_nonpos_(double x)
{
    const double kd = __dadd_rn(__fma_rn(x, 1.4426950408889634074, 6755399441055744.0), -6755399441055744.0);
    double r = __fma_rn(kd, -6.93147180369123816490e-01, x);
    r = __fma_rn(kd, -1.90821492927058770002e-10, r);
    double p = demcmc_exp_c_[13];
#pragma unroll
    for (int j = 12; j >= 0; --j) p = __fma_rn(p, r, demcmc_exp_c_[j]);
    const int k = (int)kd;
    const double scale = __hiloint2double((k + 1023) << 20, 0);
    return x < -708.0 ? 0.0 : p * scale;
}
// order-preserving 64-bit key of a double (kernels.cu: ps_key)
__device__ __forceinline__ unsigned long long demcmc_key_(double x)
{
    const unsigned long long u = (unsigned long long)__double_as_longlong(x);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double demcmc_unkey_(unsigned long long k)
{
    return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k));
}
// fixed-order CTA sum: the warp's xor tree, then the 8 warps in order; every thread gets the value
__device__ __forceinline__ double demcmc_cta_sum_(double v, double *red)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double r = red[0];
#pragma unroll
    for (int w = 1; w < 8; ++w) r += red[w];
    __syncthreads();
    return r;
}
// linearly interpolated quantile of sorted v[0..m) (numpy's and Julia's default)
__device__ __forceinline__ double demcmc_quantile_(const double *v, int m, double p)
{
    const double h = (double)(m - 1) * p;
    const int lo = (int)floor(h);
    const int hi = lo + 1 < m ? lo + 1 : lo;
    return v[lo] + (h - (double)lo) * (v[hi] - v[lo]);
}
// per label c = 1..8: first index and size of its sorted group, 1/h_c and 1/(sqrt(2 pi) M h_c) (ih = 0: no density)
struct demcmc_groups_ { int beg[9], m[9]; double ih[9], scale[9]; };

__device__ __forceinline__ int demcmc_pow2_(int M) { int p = 16; while (p < M) p <<= 1; return p; }

// the M simulations of one key into key[] / lab[] (P2 entries, dynamic shared memory), sorted by (label, value); then the
// values in place of the keys and the groups' bandwidths.  Label 255 = in no group (and the padding up to P2).
__device__ void demcmc_sim_prepare_(const double *par, unsigned sweep, unsigned unit, unsigned long long seed, int M, int n_cols,
                                    int K, unsigned long long *key, unsigned char *lab, demcmc_groups_ &g, double *red, double *sims)
{
    const int tid = threadIdx.x, P2 = demcmc_pow2_(M);
    for (int j = tid; j < P2; j += 256) {
        unsigned char l = 255;
        unsigned long long k = ~0ull;
        if (j < M) {
            demcmc_rng r;
            r.c = 0; r.unit = unit; r.sweep = sweep; r.stream = 8u + 16u * (unsigned)j;
            r.k0 = (unsigned)seed; r.k1 = (unsigned)(seed >> 32); r.has_u = 0; r.has_z = 0; r.u = 0.0; r.z = 0.0;
            double y[2] = { 0.0, 0.0 };
            demcmc_simulate(par, &r, y);
            if (sims) for (int c = 0; c < n_cols; ++c) sims[(size_t)j * n_cols + c] = y[c];
            const double val = n_cols == 2 ? y[1] : y[0];
            if (isfinite(val)) {
                if (n_cols == 1) l = 1;
                else if (y[0] >= 1.0 && y[0] <= (double)K && y[0] == floor(y[0])) l = (unsigned char)y[0];
            }
            k = demcmc_key_(val);
        }
        key[j] = k; lab[j] = l;
    }
    if (tid < 9) g.m[tid] = 0;
    __syncthreads();
    for (int size = 2; size <= P2; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = tid; t < P2 / 2; t += 256) {
                const int a = 2 * t - (t & (stride - 1)), b = a + stride;
                const bool up = (a & size) == 0;
                const unsigned char la = lab[a], lb = lab[b];
                const unsigned long long ka = key[a], kb = key[b];
                if ((la > lb || (la == lb && ka > kb)) == up) { lab[a] = lb; lab[b] = la; key[a] = kb; key[b] = ka; }
            }
            __syncthreads();
        }
    double *v = (double *)key;
    for (int j = tid; j < M; j += 256) {
        const unsigned char l = lab[j];
        if (l != 255) { atomicAdd(&g.m[l], 1); v[j] = demcmc_unkey_(key[j]); }
    }
    __syncthreads();
    if (tid == 0) { int b = 0; for (int c = 1; c <= K; ++c) { g.beg[c] = b; b += g.m[c]; } }
    __syncthreads();
    for (int c = 1; c <= K; ++c) {
        const int m = g.m[c], b = g.beg[c];
        double ih = 0.0, sc = 0.0;
        if (m >= 2) {
            double s = 0.0;
            for (int j = tid; j < m; j += 256) s += v[b + j];
            const double mean = demcmc_cta_sum_(s, red) / (double)m;
            double q = 0.0;
            for (int j = tid; j < m; j += 256) { const double dl = v[b + j] - mean; q += dl * dl; }
            const double sd = sqrt(demcmc_cta_sum_(q, red) / (double)(m - 1));
            const double iqr = demcmc_quantile_(v + b, m, 0.75) - demcmc_quantile_(v + b, m, 0.25);
            const double a = iqr > 0.0 ? fmin(sd, iqr / 1.34) : sd;
            const double h = 0.9 * a * pow((double)m, -0.2);
            if (h > 0.0 && isfinite(h)) { ih = 1.0 / h; sc = 0.39894228040143267794 / ((double)M * h); }
        }
        if (tid == 0) { g.ih[c] = ih; g.scale[c] = sc; }
    }
    __syncthreads();
}

// log-likelihood of one observation (label c, value t), computed by one whole warp: lane-strided over the group, xor tree
__device__ __forceinline__ double demcmc_sim_obs_(const double *v, const demcmc_groups_ &g, int c, double t, double floor_)
{
    const double ih = g.ih[c];
    if (!(ih > 0.0)) return log(floor_);
    const int b = g.beg[c], m = g.m[c];
    double s = 0.0;
    for (int j = (int)(threadIdx.x & 31); j < m; j += 32) {
        const double z = (t - v[b + j]) * ih;
        s += demcmc_exp_nonpos_(-0.5 * (z * z));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const double f = s * g.scale[c];
    return log(f > floor_ ? f : floor_);
}

__device__ __forceinline__ void demcmc_sim_par_(const double *th, int d, double *par)
{
#ifdef DEMCMC_NPAR
    if (threadIdx.x == 0) demcmc_prepare(th, par);
#else
    for (int k = threadIdx.x; k < d; k += 256) par[k] = th[k];
#endif
    __syncthreads();
}

// one CTA per (proposal, observation split): part[p][split] = sum of the split's ll_i.  Keys: (key_sweep[p], key_unit[p])
// when given (the test hook), else (the sweep of the entry's SweepCtx, or the eval sweep without contexts; unit_base + p)
extern "C" __global__ void __launch_bounds__(256) k_ll_sim(const double *theta, int d, const int *order, const char *ctxs, int ctx_stride,
                                                           unsigned unit_base, const unsigned *key_sweep, const unsigned *key_unit,
                                                           const double *x, int n_cols, long long n_obs, int split_len, int n_split,
                                                           double *part, unsigned long long seed, int M, int K, double floor_, double *sims)
{
    extern __shared__ unsigned long long demcmc_keys_[];
    __shared__ double par[DEMCMC_PAR_LEN_];
    __shared__ double red[8];
    __shared__ demcmc_groups_ g;
    unsigned char *lab = (unsigned char *)(demcmc_keys_ + demcmc_pow2_(M));
    const int split = blockIdx.y, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned e = order ? (unsigned)order[blockIdx.x] : blockIdx.x;
    const int p = (int)(e & 0xFFFFFFu);
    unsigned sweep, unit;
    if (key_sweep) { sweep = key_sweep[p]; unit = key_unit[p]; }
    else { sweep = ctxs ? *(const unsigned *)(ctxs + (size_t)(e >> 24) * ctx_stride) : 0xFFFFFFFFu; unit = unit_base + (unsigned)p; }
    demcmc_sim_par_(theta + (size_t)p * d, d, par);
    demcmc_sim_prepare_(par, sweep, unit, seed, M, n_cols, K, demcmc_keys_, lab, g, red,
                        (sims && split == 0) ? sims + (size_t)p * M * n_cols : nullptr);
    const double *v = (const double *)demcmc_keys_;
    const long long i0 = (long long)split * split_len, i1 = min(n_obs, i0 + (long long)split_len);
    double acc = 0.0;
    for (long long i = i0 + warp; i < i1; i += 8) {
        const double *xi = x + (size_t)i * n_cols;
        acc += demcmc_sim_obs_(v, g, n_cols == 2 ? (int)xi[0] : 1, xi[n_cols - 1], floor_);
    }
    if (lane == 0) red[warp] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += red[w];
        part[(size_t)p * n_split + split] = s;
    }
}

// demcmc_eval_pointwise / demcmc_loo: one CTA per (draw s, chunk of observations), key (eval sweep, s);
// out[o][s] = ll of observation obs0 + o
extern "C" __global__ void __launch_bounds__(256) k_ll_sim_obs(const double *theta, int d, long long n, const double *x, int n_cols,
                                                               long long obs0, long long n_obs, int chunk_len, unsigned long long seed,
                                                               int M, int K, double floor_, double *out)
{
    extern __shared__ unsigned long long demcmc_keys_[];
    __shared__ double par[DEMCMC_PAR_LEN_];
    __shared__ double red[8];
    __shared__ demcmc_groups_ g;
    unsigned char *lab = (unsigned char *)(demcmc_keys_ + demcmc_pow2_(M));
    const long long s = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    demcmc_sim_par_(theta + (size_t)s * d, d, par);
    demcmc_sim_prepare_(par, 0xFFFFFFFFu, (unsigned)s, seed, M, n_cols, K, demcmc_keys_, lab, g, red, nullptr);
    const double *v = (const double *)demcmc_keys_;
    const long long o0 = (long long)blockIdx.y * chunk_len, o1 = min(n_obs, o0 + (long long)chunk_len);
    for (long long o = o0 + warp; o < o1; o += 8) {
        const double *xi = x + (size_t)(obs0 + o) * n_cols;
        const double ll = demcmc_sim_obs_(v, g, n_cols == 2 ? (int)xi[0] : 1, xi[n_cols - 1], floor_);
        if (lane == 0) out[(size_t)o * n + s] = ll;
    }
}
)CU";

struct NvrtcApi {
    void *lib = nullptr;
    decltype(&nvrtcCreateProgram) CreateProgram = nullptr;
    decltype(&nvrtcCompileProgram) CompileProgram = nullptr;
    decltype(&nvrtcGetProgramLogSize) GetProgramLogSize = nullptr;
    decltype(&nvrtcGetProgramLog) GetProgramLog = nullptr;
    decltype(&nvrtcGetCUBINSize) GetCUBINSize = nullptr;
    decltype(&nvrtcGetCUBIN) GetCUBIN = nullptr;
    decltype(&nvrtcDestroyProgram) DestroyProgram = nullptr;
    decltype(&nvrtcGetErrorString) GetErrorString = nullptr;
};
static NvrtcApi g_nvrtc;
static std::mutex g_custom_mu;                                   // the NVRTC table and the cubin cache
static std::map<std::pair<int, std::string>, std::string> g_custom_cubin;   // (1 = simulator, source text) -> sm_100a cubin

static int nvrtc_load()                                          // under g_custom_mu
{
    if (g_nvrtc.lib) return 0;
    void *lib = dlopen("libnvrtc.so.12", RTLD_NOW | RTLD_LOCAL);
    if (!lib) { g_be_err = std::string("custom likelihoods need NVRTC: cannot load libnvrtc.so.12: ") + dlerror(); return -2; }
#define SYM(field, sym) do { *(void **)(&g_nvrtc.field) = dlsym(lib, sym); if (!g_nvrtc.field) { g_be_err = std::string("libnvrtc misses ") + sym; dlclose(lib); return -2; } } while (0)
    SYM(CreateProgram, "nvrtcCreateProgram"); SYM(CompileProgram, "nvrtcCompileProgram");
    SYM(GetProgramLogSize, "nvrtcGetProgramLogSize"); SYM(GetProgramLog, "nvrtcGetProgramLog");
    SYM(GetCUBINSize, "nvrtcGetCUBINSize"); SYM(GetCUBIN, "nvrtcGetCUBIN");
    SYM(DestroyProgram, "nvrtcDestroyProgram"); SYM(GetErrorString, "nvrtcGetErrorString");
#undef SYM
    g_nvrtc.lib = lib;
    return 0;
}

// the cubin of a custom (sim = 0) or simulator (sim = 1) `source`, compiled on the first request (under g_custom_mu)
static int custom_cubin(const char *source, const std::string **cubin, int sim = 0)
{
    const std::pair<int, std::string> key(sim, source);
    auto it = g_custom_cubin.find(key);
    if (it != g_custom_cubin.end()) { *cubin = &it->second; return 0; }
    if (int rc = nvrtc_load()) return rc;
    const std::string text = sim ? std::string(SIM_PRELUDE) + source + "\n" + SIM_KERNEL : std::string(CUSTOM_PRELUDE) + source + "\n" + CUSTOM_KERNEL;
    nvrtcProgram prog = nullptr;
    nvrtcResult r = g_nvrtc.CreateProgram(&prog, text.c_str(), "demcmc_custom.cu", 0, nullptr, nullptr);
    if (r != NVRTC_SUCCESS) { g_be_err = std::string("nvrtcCreateProgram: ") + g_nvrtc.GetErrorString(r); return -1; }
    // --fmad=false: the library's own arithmetic (csrc/Makefile) and the reference's, without contraction
    const char *opts[] = { "-arch=sm_100a", "-std=c++17", "--fmad=false" };
    r = g_nvrtc.CompileProgram(prog, 3, opts);
    if (r != NVRTC_SUCCESS) {
        size_t n = 0;
        std::string log;
        if (g_nvrtc.GetProgramLogSize(prog, &n) == NVRTC_SUCCESS && n > 1) { log.resize(n); g_nvrtc.GetProgramLog(prog, &log[0]); log.resize(n - 1); }
        g_nvrtc.DestroyProgram(&prog);
        g_be_err = std::string(sim ? "simulator" : "custom likelihood") + " does not compile (" + std::string(g_nvrtc.GetErrorString(r)) + "):\n" + log;
        return log.find("DEMCMC_NPAR is above") != std::string::npos ? -2 : -1;
    }
    size_t n = 0;
    std::string bin;
    r = g_nvrtc.GetCUBINSize(prog, &n);
    if (r == NVRTC_SUCCESS) { bin.resize(n); r = g_nvrtc.GetCUBIN(prog, &bin[0]); }
    g_nvrtc.DestroyProgram(&prog);
    if (r != NVRTC_SUCCESS) { g_be_err = std::string("nvrtcGetCUBIN: ") + g_nvrtc.GetErrorString(r); return -1; }
    *cubin = &(g_custom_cubin[key] = std::move(bin));
    return 0;
}

int custom_compile(const char *source)
{
    std::lock_guard<std::mutex> lk(g_custom_mu);
    const std::string *cubin = nullptr;
    return custom_cubin(source, &cubin);
}

struct CustomModule { cudaLibrary_t lib; cudaKernel_t kernel, obs_kernel; int npar; };

int custom_load(const char *source, void **module, int *has_obs)
{
    *module = nullptr;
    std::string cubin;
    {
        std::lock_guard<std::mutex> lk(g_custom_mu);
        const std::string *c = nullptr;
        if (int rc = custom_cubin(source, &c)) return rc;
        cubin = *c;
    }
    CustomModule *mod = new CustomModule();
    cudaError_t e = cudaLibraryLoadData(&mod->lib, cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0);
    if (e != cudaSuccess) { delete mod; cu_fail(e, "cudaLibraryLoadData (custom likelihood)"); return -3; }
    e = cudaLibraryGetKernel(&mod->kernel, mod->lib, "k_ll_custom");
    void *flag = nullptr;
    size_t bytes = 0;
    if (e == cudaSuccess) e = cudaLibraryGetGlobal(&flag, &bytes, mod->lib, "demcmc_custom_has_obs");
    if (e == cudaSuccess) e = cudaMemcpy(has_obs, flag, sizeof(int), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaLibraryGetKernel(&mod->obs_kernel, mod->lib, "k_ll_custom_obs");
    if (e == cudaSuccess) e = cudaLibraryGetGlobal(&flag, &bytes, mod->lib, "demcmc_custom_npar");
    if (e == cudaSuccess) e = cudaMemcpy(&mod->npar, flag, sizeof(int), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) { cudaLibraryUnload(mod->lib); delete mod; cu_fail(e, "loading k_ll_custom"); return -3; }
    *module = mod;
    return 0;
}

void custom_unload(void *module)
{
    if (!module) return;
    CustomModule *mod = (CustomModule *)module;
    cudaLibraryUnload(mod->lib);
    delete mod;
}

int sim_compile(const char *source)
{
    std::lock_guard<std::mutex> lk(g_custom_mu);
    const std::string *cubin = nullptr;
    return custom_cubin(source, &cubin, 1);
}

// a simulator module: k_ll_sim as CustomModule.kernel, k_ll_sim_obs as obs_kernel
int sim_load(const char *source, void **module)
{
    *module = nullptr;
    std::string cubin;
    {
        std::lock_guard<std::mutex> lk(g_custom_mu);
        const std::string *c = nullptr;
        if (int rc = custom_cubin(source, &c, 1)) return rc;
        cubin = *c;
    }
    CustomModule *mod = new CustomModule();
    cudaError_t e = cudaLibraryLoadData(&mod->lib, cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0);
    if (e != cudaSuccess) { delete mod; cu_fail(e, "cudaLibraryLoadData (simulator)"); return -3; }
    e = cudaLibraryGetKernel(&mod->kernel, mod->lib, "k_ll_sim");
    if (e == cudaSuccess) e = cudaLibraryGetKernel(&mod->obs_kernel, mod->lib, "k_ll_sim_obs");
    const size_t smem = sim_smem(SIM_MAX_DRAWS);
    if (e == cudaSuccess) e = cudaFuncSetAttribute((const void *)mod->kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute((const void *)mod->obs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { cudaLibraryUnload(mod->lib); delete mod; cu_fail(e, "loading k_ll_sim"); return -3; }
    *module = mod;
    return 0;
}

// k_ll_sim over the entries of lv; keys from key_sweep / key_unit (device, [lv.n]) when given
static int launch_ll_sim(const ConfigDev &cfg, const ModelDev &m, const double *theta, const Level &lv, const uint32_t *key_sweep,
                         const uint32_t *key_unit, double *ll_part, double *sims)
{
    if (!m.custom) { g_be_err = "simulator not loaded"; return -1; }
    const CustomModule *mod = (const CustomModule *)m.custom;
    int d = m.d, n_cols = m.n_cols, split_len = m.split_len, n_split = m.n_osplit, M = m.n_sim, K = m.n_lab;
    int ctx_stride = (int)sizeof(SweepCtx);
    unsigned unit_base = (unsigned)(cfg.group_begin * cfg.Np);
    long long n_obs = m.n_obs;
    unsigned long long seed = m.sim_seed;
    double floor_ = m.sim_floor;
    const int *order = lv.order;
    const char *ctxs = (const char *)lv.ctxs;
    const double *x = m.x;
    void *args[] = { &theta, &d, &order, &ctxs, &ctx_stride, &unit_base, &key_sweep, &key_unit, &x, &n_cols, &n_obs, &split_len, &n_split,
                     &ll_part, &seed, &M, &K, &floor_, &sims };
    CU(cudaLaunchKernel((const void *)mod->kernel, dim3((unsigned)lv.n, (unsigned)n_split), dim3(256), args, sim_smem(M), stream()));
    LAUNCHED("k_ll_sim");
    return 0;
}

static int launch_ll_custom(const ModelDev &m, const double *theta, const Level &lv, double *ll_part)
{
    if (!m.custom) { g_be_err = "custom likelihood not loaded"; return -1; }
    const CustomModule *mod = (const CustomModule *)m.custom;
    int d = m.d, n = lv.n, n_cols = m.n_cols, split_len = m.split_len, n_split = m.n_osplit * m.n_ksplit;
    long long n_obs = m.n_obs;
    const int *order = lv.order;
    const double *x = m.x;
    void *args[] = { &theta, &d, &order, &n, &x, &n_cols, &n_obs, &split_len, &n_split, &ll_part };
    CU(cudaLaunchKernel((const void *)mod->kernel, dim3((lv.n + PW_TP - 1) / PW_TP, n_split), dim3(PW_THREADS), args, 0, stream()));
    LAUNCHED("k_ll_custom");
    return 0;
}

int launch_loglik(const ConfigDev &cfg, const ModelDev &m, const double *theta, const Level &lv, double *ll_part, long long *ll_acc)
{
    (void)cfg;
    if (lv.n <= 0 || m.kind == M_BINOMIAL || m.kind == M_RASTRIGIN) return 0;
    if (is_ssd(m.kind)) {
        // the proposal kernel of this level has staged the centred means and cleared the accumulators
        const XdStage &xs = g_xs[g_dev][g_lane];
        if (!xs.bfrag || !xs.magic) { g_be_err = "mean staging buffer missing"; return -1; }
        return launch_xdot(m, xs, lv, ll_acc);
    }
    if (m.kind == M_CUSTOM) return launch_ll_custom(m, theta, lv, ll_part);
    if (m.kind == M_SIMULATED) return launch_ll_sim(cfg, m, theta, lv, nullptr, nullptr, ll_part, nullptr);
    dim3 grid((lv.n + PW_TP - 1) / PW_TP, m.n_osplit);
    if (m.kind == M_GAUSSIAN) k_ll_pointwise<M_GAUSSIAN><<<grid, PW_THREADS, 0, stream()>>>(m, theta, lv, ll_part);
    else if (m.kind == M_LNR) k_ll_pointwise<M_LNR><<<grid, PW_THREADS, 0, stream()>>>(m, theta, lv, ll_part);
    else if (m.kind == M_LBA) k_ll_pointwise<M_LBA><<<grid, PW_THREADS, 0, stream()>>>(m, theta, lv, ll_part);
    else { g_be_err = "no kernel for this model kind"; return -1; }
    LAUNCHED("k_ll_pointwise");
    return 0;
}

// ------------------------------------------------------------------------------------------------
// data packing for k_xdot: x[n][k] (MVN, observation-major) or y[k][n] (hierarchical,
// subject-major) -> center[k], then the centred data as DMMA A fragments (de_types.h:
// ssd_pack_index), zero padded; also sum x'^2 and max_i |x'_i|.  Fixed reduction order.
// ------------------------------------------------------------------------------------------------
__device__ double block_sum_256(double v, double *red)
{
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
    if (threadIdx.x == 0) { for (int w = 0; w < 8; ++w) s += red[w]; red[8] = s; }
    __syncthreads();
    s = red[8];
    __syncthreads();
    return s;
}

__global__ void __launch_bounds__(256) k_col_center(const double *x, double *center, int64_t n, int k, int obs_major)
{
    __shared__ double red[9];
    const int kk = blockIdx.x;
    double s = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += 256) s += obs_major ? x[i * k + kk] : x[(int64_t)kk * n + i];
    const double c = n > 0 ? block_sum_256(s, red) / (double)n : 0.0;
    if (threadIdx.x == 0) center[kk] = c;
}

// one thread per observation: writes its centred row into the packed layout; per block the sum and
// the maximum of the squared row norms
__global__ void __launch_bounds__(256) k_pack_rows(const double *x, const double *center, double *xp, double *blk_sq, double *blk_max,
                                                   int64_t n, int k, int ksplit_len, int nj, int64_t n_tiles, int obs_major, int half, int corrupt)
{
    __shared__ double red[9];
    __shared__ double redm[8];
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    double q = 0.0;
    if (i < n)
        for (int kk = 0; kk < k; ++kk) {
            const double v = (obs_major ? x[i * k + kk] : x[(int64_t)kk * n + i]) - center[kk];
            q += v * v;
            // (mutation test 2: the second row tile of a pair packs its half k-step over the first tile's)
            const int64_t ip = (corrupt == 2 && half && (kk % ksplit_len) / 4 == nj - 1) ? (i & ~(int64_t)8) : i;
            xp[ssd_pack_index(ip, kk, ksplit_len, nj, n_tiles, half)] = v;
        }
    double mx = q;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) redm[threadIdx.x >> 5] = mx;
    const double s = block_sum_256(q, red);
    if (threadIdx.x == 0) {
        double mm = redm[0];
        for (int w = 1; w < 8; ++w) mm = fmax(mm, redm[w]);
        blk_sq[blockIdx.x] = s;
        blk_max[blockIdx.x] = mm;
    }
}

size_t pack_ssd_doubles(const ModelDev &m) { return (size_t)m.n_ksplit * (size_t)(m.ssd_ld / SSD_TN) * m.ssd_nj * 256; }

int launch_pack_ssd(const double *x_in, int in_on_device, const double *center_host, ModelDev *m)
{
    const size_t bytes = sizeof(double) * (size_t)m->ssd_n * m->ssd_k;
    const int n_blk = (int)std::max<int64_t>(1, (m->ssd_n + 255) / 256);
    const double *src = x_in;
    double *tmp = nullptr, *blk = (double *)dmalloc(sizeof(double) * 2 * n_blk);
    if (!blk) return -1;
    if (!in_on_device) {
        tmp = (double *)dmalloc(bytes);
        if (!tmp) { dfree(blk); return -1; }
        if (h2d(tmp, x_in, bytes)) { dfree(tmp); dfree(blk); return -1; }
        src = tmp;
    }
    const int obs_major = m->kind == M_HIER ? 0 : 1;
    cudaError_t e = cudaMemsetAsync(const_cast<double *>(m->xT), 0, sizeof(double) * pack_ssd_doubles(*m), stream());
    if (e == cudaSuccess) e = cudaMemsetAsync(blk, 0, sizeof(double) * 2 * n_blk, stream());
    if (e == cudaSuccess && center_host) e = cudaMemcpyAsync(const_cast<double *>(m->center), center_host, sizeof(double) * m->ssd_k, cudaMemcpyHostToDevice, stream());
    if (e == cudaSuccess) {
        if (!center_host) k_col_center<<<m->ssd_k, 256, 0, stream()>>>(src, const_cast<double *>(m->center), m->ssd_n, m->ssd_k, obs_major);
        k_pack_rows<<<n_blk, 256, 0, stream()>>>(src, m->center, const_cast<double *>(m->xT), blk, blk + n_blk, m->ssd_n, m->ssd_k,
                                                 m->ksplit_len, m->ssd_nj, m->ssd_ld / SSD_TN, obs_major, m->ssd_half, m->debug_corrupt);
        g_launches += 2;
        e = cudaGetLastError();
    }
    std::vector<double> h(2 * (size_t)n_blk);
    if (e == cudaSuccess) e = cudaMemcpyAsync(h.data(), blk, sizeof(double) * 2 * n_blk, cudaMemcpyDeviceToHost, stream());
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream());
    double xx = 0.0, mx = 0.0;
    for (int b = 0; b < n_blk; ++b) { xx += h[b]; mx = std::max(mx, h[n_blk + b]); }
    m->ssd_xx = xx;
    m->ssd_rowmax = 2.0 * sqrt(mx);                          // a chain of k_xdot sums the terms of TWO observation rows
    dfree(tmp); dfree(blk);
    if (e != cudaSuccess) return cu_fail(e, "k_pack_rows");
    return 0;
}

// ------------------------------------------------------------------------------------------------
// evaluation of arbitrary parameter vectors (init_particle weights, demcmc_eval)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(PA_THREADS) k_eval_finish(ConfigDev cfg, ModelDev m, const double *theta, int64_t n,
                                                             const double *part, const long long *acc, const double *q,
                                                             double *ll, double *prior, double *w, double *xdot)
{
    const int64_t wi = ((int64_t)blockIdx.x * PA_THREADS + threadIdx.x) >> 5;
    if (wi >= n) return;
    const WarpLanes co;
    const double *th = theta + (size_t)wi * cfg.d;
    bool inb; double pr;
    bounds_and_prior(co, cfg, m, th, inb, pr);
    const int n_split = m.n_osplit * m.n_ksplit;
    double s = 0.0;
    if (is_ssd(m.kind)) s = (double)acc[wi] * q[wi];
    else {
        if (m.kind != M_BINOMIAL && m.kind != M_RASTRIGIN) for (int c = co.lane(); c < n_split; c += 32) s += part[(size_t)wi * n_split + c];
        s = co.sum(s);
    }
    const double l = finalize_ll(m, th, s, mean_sq(co, m, th));
    if (co.lane() == 0) {
        if (ll) ll[wi] = l;
        if (xdot) xdot[wi] = s;
        if (prior) prior[wi] = inb ? pr : -inf();
        if (w) w[wi] = cfg.fitness == FITNESS_FUN ? (inb ? l : (cfg.update == UPDATE_MAXIMIZE ? -inf() : inf())) : (inb ? add(pr, l) : -inf());
    }
}

int launch_eval(const ConfigDev &cfg, const ModelDev &m, const double *theta, int64_t n, double *ll, double *prior,
                double *w, double *scratch_part, double *xdot)
{
    if (n <= 0) return 0;
    Level lv; lv.order = nullptr; lv.n = (int32_t)n; lv.ctxs = nullptr;
    const int blocks = (int)((n * 32 + PA_THREADS - 1) / PA_THREADS);
    long long *acc = nullptr;
    double *q = nullptr;
    if (is_ssd(m.kind)) {
        XdStage *xs = xd_stage(m, (int)n);
        if (!xs) return -1;
        acc = (long long *)dmalloc(sizeof(long long) * n);
        q = (double *)dmalloc(sizeof(double) * n);
        if (!acc || !q) { dfree(acc); dfree(q); return -1; }
        k_stage_means<<<blocks, PA_THREADS, 0, stream()>>>(m, theta, n, xs->bfrag, xs->magic, acc, q);
        LAUNCHED("k_stage_means");
        if (launch_xdot(m, *xs, lv, acc)) { dfree(acc); dfree(q); return -1; }
    } else if (launch_loglik(cfg, m, theta, lv, scratch_part, nullptr)) return -1;
    k_eval_finish<<<blocks, PA_THREADS, 0, stream()>>>(cfg, m, theta, n, scratch_part, acc, q, ll, prior, w, xdot);
    LAUNCHED("k_eval_finish");
    if (acc) { cudaStreamSynchronize(stream()); dfree(acc); dfree(q); }
    return 0;
}

int launch_eval_sim(const ConfigDev &cfg, const ModelDev &m, const double *theta, int64_t n, const uint32_t *sweep, const uint32_t *unit,
                    double *ll, double *prior, double *sims, double *scratch_part)
{
    if (n <= 0) return 0;
    Level lv; lv.order = nullptr; lv.n = (int32_t)n; lv.ctxs = nullptr;
    if (launch_ll_sim(cfg, m, theta, lv, sweep, unit, scratch_part, sims)) return -1;
    const int blocks = (int)((n * 32 + PA_THREADS - 1) / PA_THREADS);
    k_eval_finish<<<blocks, PA_THREADS, 0, stream()>>>(cfg, m, theta, n, scratch_part, nullptr, nullptr, ll, prior, nullptr, nullptr);
    LAUNCHED("k_eval_finish");
    return 0;
}

// ------------------------------------------------------------------------------------------------
// model comparison (demcmc_eval_pointwise / demcmc_loo)
//   k_ll_obs<KIND>  the pointwise matrix out[obs][draw] of a tile of 32 draws (one per lane) x 64 observations (8 per
//                   warp): every density is the per-observation function the summed likelihood uses (de_math.h), so a
//                   warp reads one observation (a broadcast) and writes 32 consecutive doubles.  The streamed kinds take
//                   the centred data x' from the packed xT and the centred means from k_ll_obs_prep, and form
//                   |x'_i - m'|^2 directly on the CUDA cores.
//   k_psis          one CTA per observation, its S values in dynamic shared memory: max / min / sums, a radix select of
//                   the cutoff on order-preserving 64-bit keys, a bitonic sort of the tail, the GPD fit with its m x M
//                   log1p terms split over the warps, the smoothing and the four outputs.  Every reduction runs in a
//                   fixed order (per thread, warp tree, warps in order), so the outputs do not depend on the launch.
// ------------------------------------------------------------------------------------------------
constexpr int OB_TD = 32;            // draws per CTA, one per lane
constexpr int OB_TO = 64;            // observations per CTA, 8 per warp
constexpr int OB_THREADS = 256;
constexpr int OB_KC = 32;            // dimensions of the streamed kinds staged per step

// the streamed kinds: centred means transposed, mt[k][n] (lanes read consecutive draws), and the per-draw constants
__global__ void __launch_bounds__(256) k_ll_obs_prep(ModelDev m, const double *theta, int64_t n, double *mt, double *c0, double *s2)
{
    const int64_t t = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (t >= n * m.ssd_k) return;
    const int k = (int)(t / n);
    const int64_t s = t - (int64_t)k * n;
    const double *th = theta + (size_t)s * m.d;
    mt[t] = centred_mean(m, th, k);
    if (k == 0) ssd_obs_const(m, th, c0[s], s2[s]);
}

template <int KIND>
__global__ void __launch_bounds__(OB_THREADS) k_ll_obs(const __grid_constant__ ModelDev m, const double *theta, int64_t n, int64_t obs0,
                                                      int64_t n_obs, const double *mt, const double *c0, const double *s2, double *out)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t s0 = (int64_t)blockIdx.y * OB_TD, i0 = (int64_t)blockIdx.x * OB_TO;
    const int64_t s = s0 + lane;
    const int no = (int)min((int64_t)OB_TO, n_obs - i0);
    const int64_t n_tiles = m.ssd_ld / SSD_TN;
    if (KIND == M_MVNORMAL || KIND == M_MVN_FULL) {
        __shared__ double xs[OB_TO][OB_KC + 1];
        __shared__ double ms[OB_KC][OB_TD];
        double acc[OB_TO / 8];
#pragma unroll
        for (int q = 0; q < OB_TO / 8; ++q) acc[q] = 0.0;
        for (int k0 = 0; k0 < m.ssd_k; k0 += OB_KC) {
            const int kc = min(OB_KC, m.ssd_k - k0);
            __syncthreads();
            for (int e = threadIdx.x; e < OB_TO * OB_KC; e += OB_THREADS) {
                const int o = e / OB_KC, k = e % OB_KC;
                xs[o][k] = (o < no && k < kc) ? m.xT[ssd_pack_index(obs0 + i0 + o, k0 + k, m.ksplit_len, m.ssd_nj, n_tiles, m.ssd_half)] : 0.0;
            }
            for (int e = threadIdx.x; e < OB_KC * OB_TD; e += OB_THREADS) {
                const int k = e / OB_TD, t = e % OB_TD;
                ms[k][t] = (k < kc && s0 + t < n) ? mt[(size_t)(k0 + k) * n + s0 + t] : 0.0;
            }
            __syncthreads();
            for (int k = 0; k < kc; ++k) {
                const double mk = ms[k][lane];
#pragma unroll
                for (int q = 0; q < OB_TO / 8; ++q) { const double dl = xs[warp + 8 * q][k] - mk; acc[q] = __fma_rn(dl, dl, acc[q]); }
            }
        }
        if (s >= n) return;
        const double a = c0[s], b = s2[s];
#pragma unroll
        for (int q = 0; q < OB_TO / 8; ++q) {
            const int o = warp + 8 * q;
            if (o < no) out[(size_t)(i0 + o) * n + s] = ssd_obs_ll(a, b, acc[q]);
        }
    } else if (KIND == M_HIER) {
        if (s >= n) return;
        const double a = c0[s], b = s2[s];
        for (int o = warp; o < no; o += 8) {
            const int64_t i = obs0 + i0 + o;
            const int subj = (int)(i / m.n_per);
            const double dl = m.xT[ssd_pack_index(i - (int64_t)subj * m.n_per, subj, m.ksplit_len, m.ssd_nj, n_tiles, m.ssd_half)] -
                              mt[(size_t)subj * n + s];
            out[(size_t)(i0 + o) * n + s] = ssd_obs_ll(a, b, dl * dl);
        }
    } else if (KIND == M_BINOMIAL) {
        if (s < n && warp == 0) out[s] = binomial_ll(m.binom_N, m.binom_k, theta[(size_t)s * m.d]);
    } else {
        __shared__ double par[OB_TD][MAX_ACC + 5];
        if (threadIdx.x < OB_TD && s0 + threadIdx.x < n) pointwise_par<KIND>(m, theta + (size_t)(s0 + threadIdx.x) * m.d, par[threadIdx.x]);
        __syncthreads();
        if (s >= n) return;
        const double *sg = m.has_sigma ? m.sigma_acc : nullptr;
        for (int o = warp; o < no; o += 8) {
            const int64_t i = obs0 + i0 + o;
            const double x = m.x[i];
            double v;
            if (KIND == M_GAUSSIAN) v = gaussian_obs(par[lane], x);
            else if (KIND == M_LNR) v = lnr_obs(par[lane], m.n_dim, sg, x, m.choice[i] - 1);
            else v = lba_obs(par[lane], m.n_dim, par[lane][m.n_dim + 3], m.lba_floor, x, m.choice[i] - 1);
            out[(size_t)(i0 + o) * n + s] = v;
        }
    }
}

static int launch_ll_custom_obs(const ModelDev &m, const double *theta, int64_t n, int64_t obs0, int64_t n_obs, double *out)
{
    if (!m.custom) { g_be_err = "custom likelihood not loaded"; return -1; }
    const CustomModule *mod = (const CustomModule *)m.custom;
    const size_t smem = sizeof(double) * OB_TD * (size_t)((mod->npar > 0 ? mod->npar : m.d) | 1);
    CU(cudaFuncSetAttribute((const void *)mod->obs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int d = m.d, n_cols = m.n_cols;
    long long nn = n, o0 = obs0, no = n_obs;
    const double *x = m.x;
    void *args[] = { &theta, &d, &nn, &x, &n_cols, &o0, &no, &out };
    CU(cudaLaunchKernel((const void *)mod->obs_kernel, dim3((unsigned)((n_obs + OB_TO - 1) / OB_TO), (unsigned)((n + OB_TD - 1) / OB_TD)),
                        dim3(OB_THREADS), args, smem, stream()));
    LAUNCHED("k_ll_custom_obs");
    return 0;
}

static int launch_ll_sim_obs(const ModelDev &m, const double *theta, int64_t n, int64_t obs0, int64_t n_obs, double *out)
{
    if (!m.custom) { g_be_err = "simulator not loaded"; return -1; }
    const CustomModule *mod = (const CustomModule *)m.custom;
    int d = m.d, n_cols = m.n_cols, chunk_len = m.split_len, M = m.n_sim, K = m.n_lab;
    long long nn = n, o0 = obs0, no = n_obs;
    unsigned long long seed = m.sim_seed;
    double floor_ = m.sim_floor;
    const double *x = m.x;
    const int64_t n_chunks = (n_obs + chunk_len - 1) / chunk_len;
    if (n_chunks > 65535) { g_be_err = "too many observations for one k_ll_sim_obs launch"; return -1; }
    void *args[] = { &theta, &d, &nn, &x, &n_cols, &o0, &no, &chunk_len, &seed, &M, &K, &floor_, &out };
    CU(cudaLaunchKernel((const void *)mod->obs_kernel, dim3((unsigned)n, (unsigned)n_chunks), dim3(256), args, sim_smem(M), stream()));
    LAUNCHED("k_ll_sim_obs");
    return 0;
}

int launch_pointwise(const ModelDev &m, const double *theta, int64_t n, int64_t obs0, int64_t n_obs, double *out)
{
    if (n <= 0 || n_obs <= 0) return 0;
    if (n > (int64_t)65535 * OB_TD) { g_be_err = "too many draws for one pointwise launch"; return -1; }
    if (m.kind == M_CUSTOM) return launch_ll_custom_obs(m, theta, n, obs0, n_obs, out);
    if (m.kind == M_SIMULATED) return launch_ll_sim_obs(m, theta, n, obs0, n_obs, out);
    const dim3 grid((unsigned)((n_obs + OB_TO - 1) / OB_TO), (unsigned)((n + OB_TD - 1) / OB_TD));
    double *mt = nullptr, *c0 = nullptr, *s2 = nullptr;
    if (is_ssd(m.kind)) {
        mt = (double *)dmalloc(sizeof(double) * (size_t)n * m.ssd_k);
        c0 = (double *)dmalloc(sizeof(double) * (size_t)n);
        s2 = (double *)dmalloc(sizeof(double) * (size_t)n);
        if (!mt || !c0 || !s2) { dfree(mt); dfree(c0); dfree(s2); return -1; }
        k_ll_obs_prep<<<(unsigned)((n * m.ssd_k + 255) / 256), 256, 0, stream()>>>(m, theta, n, mt, c0, s2);
        ++g_launches;
    }
    switch (m.kind) {
    case M_GAUSSIAN: k_ll_obs<M_GAUSSIAN><<<grid, OB_THREADS, 0, stream()>>>(m, theta, n, obs0, n_obs, mt, c0, s2, out); break;
    case M_LNR: k_ll_obs<M_LNR><<<grid, OB_THREADS, 0, stream()>>>(m, theta, n, obs0, n_obs, mt, c0, s2, out); break;
    case M_LBA: k_ll_obs<M_LBA><<<grid, OB_THREADS, 0, stream()>>>(m, theta, n, obs0, n_obs, mt, c0, s2, out); break;
    case M_BINOMIAL: k_ll_obs<M_BINOMIAL><<<grid, OB_THREADS, 0, stream()>>>(m, theta, n, obs0, n_obs, mt, c0, s2, out); break;
    case M_MVNORMAL: k_ll_obs<M_MVNORMAL><<<grid, OB_THREADS, 0, stream()>>>(m, theta, n, obs0, n_obs, mt, c0, s2, out); break;
    case M_MVN_FULL: k_ll_obs<M_MVN_FULL><<<grid, OB_THREADS, 0, stream()>>>(m, theta, n, obs0, n_obs, mt, c0, s2, out); break;
    case M_HIER: k_ll_obs<M_HIER><<<grid, OB_THREADS, 0, stream()>>>(m, theta, n, obs0, n_obs, mt, c0, s2, out); break;
    default: dfree(mt); dfree(c0); dfree(s2); g_be_err = "no pointwise kernel for this model kind"; return -1;
    }
    const cudaError_t e = cudaGetLastError();
    ++g_launches;
    dfree(mt); dfree(c0); dfree(s2);                 // stream-ordered: freed after the kernel has run
    if (e != cudaSuccess) return cu_fail(e, "k_ll_obs");
    return 0;
}

// ---- k_psis -------------------------------------------------------------------------------------
constexpr int PS_THREADS = 256;
constexpr int PS_WARPS = PS_THREADS / 32;
constexpr int PS_MAX_GRID = 64;      // >= 30 + floor(sqrt(PSIS_MAX_TAIL))

// fixed-order block reductions: per thread, then the warp's xor tree, then the warps in order (every thread forms the same
// value from the same eight partials)
struct PsSum { __device__ __forceinline__ double operator()(double a, double b) const { return a + b; } };
struct PsMax { __device__ __forceinline__ double operator()(double a, double b) const { return fmax(a, b); } };
struct PsMin { __device__ __forceinline__ double operator()(double a, double b) const { return fmin(a, b); } };
template <class Op>
__device__ __forceinline__ double ps_reduce(double v, double *red, Op op)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = op(v, __shfl_xor_sync(0xffffffffu, v, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double r = red[0];
#pragma unroll
    for (int w = 1; w < PS_WARPS; ++w) r = op(r, red[w]);
    __syncthreads();
    return r;
}
// order-preserving 64-bit key of a double (larger value, larger key)
__device__ __forceinline__ unsigned long long ps_key(double x)
{
    const unsigned long long u = (unsigned long long)__double_as_longlong(x);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double ps_unkey(unsigned long long k)
{
    return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k));
}

__global__ void __launch_bounds__(PS_THREADS) k_psis(const double *ll, int S, double *elpd_out, double *k_out, double *lppd_out, double *pw_out)
{
    extern __shared__ double v[];                   // [S] the observation's log-likelihoods
    __shared__ double tv[PSIS_MAX_TAIL];            // tail: log ratio (then its smoothed value) ...
    __shared__ int ti[PSIS_MAX_TAIL];               // ... and its draw
    __shared__ double ty[PSIS_MAX_TAIL];            // exp(x) - exp(cutoff)
    __shared__ double gb[PS_MAX_GRID], gl[PS_MAX_GRID], gw[PS_MAX_GRID];
    __shared__ unsigned hist[256];
    __shared__ double red[PS_WARPS];
    __shared__ int sh_digit, sh_rank, sh_nt;
    __shared__ double sh_b;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const size_t obs = blockIdx.x;
    const double *src = ll + obs * (size_t)S;
    bool fin = true;
    double mn = HUGE_VAL, mx = -HUGE_VAL, sum = 0.0;
    for (int s = tid; s < S; s += PS_THREADS) { const double a = src[s]; v[s] = a; fin = fin && isfinite(a); mn = fmin(mn, a); mx = fmax(mx, a); sum += a; }
    if (!__syncthreads_and(fin)) {
        if (tid == 0) { const double q = qnan(); elpd_out[obs] = q; k_out[obs] = q; lppd_out[obs] = q; pw_out[obs] = q; }
        return;
    }
    mn = ps_reduce(mn, red, PsMin());
    mx = ps_reduce(mx, red, PsMax());
    sum = ps_reduce(sum, red, PsSum());
    double e = 0.0, q = 0.0;
    const double mean = sum / (double)S;
    for (int s = tid; s < S; s += PS_THREADS) { const double a = v[s]; e += exp(a - mx); const double dl = a - mean; q += dl * dl; }
    e = ps_reduce(e, red, PsSum());
    q = ps_reduce(q, red, PsSum());
    // (M+1)-th largest log ratio x_s = mn - ll_s (= -ll_s - max(-ll)): MSB-first radix select, 8 bits a pass
    const int M = psis_tail_len(S);
    unsigned long long prefix = 0, mask = 0;
    int rank = M + 1;
    for (int shift = 56; shift >= 0; shift -= 8) {
        hist[tid] = 0;
        __syncthreads();
        for (int s = tid; s < S; s += PS_THREADS) {
            const unsigned long long k = ps_key(mn - v[s]);
            if ((k & mask) == prefix) atomicAdd(&hist[(k >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (warp == 0) {                            // lane L holds bins 255 - 8L .. 248 - 8L, counted from the top
            int c[8], tot = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) { c[j] = (int)hist[255 - 8 * lane - j]; tot += c[j]; }
            int inc = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += y; }
            const int exc = inc - tot;
            if (exc < rank && rank <= inc) {
                int a = exc;
                for (int j = 0; j < 8; ++j) {
                    if (a + c[j] >= rank) { sh_digit = 255 - 8 * lane - j; sh_rank = rank - a; break; }
                    a += c[j];
                }
            }
        }
        __syncthreads();
        prefix |= (unsigned long long)sh_digit << shift;
        mask |= 0xFFull << shift;
        rank = sh_rank;
    }
    const double cutoff = fmax(ps_unkey(prefix), DE_LOG_DBL_MIN);
    // the tail, sorted by (x, draw): padding sorts last
    if (tid == 0) sh_nt = 0;
    for (int j = tid; j < PSIS_MAX_TAIL; j += PS_THREADS) { tv[j] = HUGE_VAL; ti[j] = 0x7fffffff; }
    __syncthreads();
    for (int s = tid; s < S; s += PS_THREADS) {
        const double x = mn - v[s];
        if (x > cutoff) { const int j = atomicAdd(&sh_nt, 1); tv[j] = x; ti[j] = s; }
    }
    __syncthreads();
    const int nt = sh_nt;
    for (int size = 2; size <= PSIS_MAX_TAIL; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = tid; t < PSIS_MAX_TAIL / 2; t += PS_THREADS) {
                const int a = 2 * t - (t & (stride - 1)), b = a + stride;
                const bool up = (a & size) == 0;
                const bool gt = tv[a] > tv[b] || (tv[a] == tv[b] && ti[a] > ti[b]);
                if (gt == up) { const double x = tv[a]; tv[a] = tv[b]; tv[b] = x; const int i = ti[a]; ti[a] = ti[b]; ti[b] = i; }
            }
            __syncthreads();
        }
    double khat = HUGE_VAL;
    if (nt > 4) {
        const double ec = exp(cutoff);
        for (int j = tid; j < nt; j += PS_THREADS) ty[j] = exp(tv[j]) - ec;
        __syncthreads();
        const int m = gpd_grid_len(nt);
        const double yq = ty[gpd_quartile_index(nt)], ymax = ty[nt - 1];
        for (int g = warp; g < m; g += PS_WARPS) {
            const double b = gpd_grid_b(g, m, yq, ymax);
            double a = 0.0;
            for (int j = lane; j < nt; j += 32) a += log1p(-b * ty[j]);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
            if (lane == 0) { gb[g] = b; gl[g] = gpd_profile(b, a / (double)nt, nt); }
        }
        __syncthreads();
        if (tid < m) {
            double a = 0.0;
            for (int h = 0; h < m; ++h) a += exp(gl[h] - gl[tid]);
            gw[tid] = 1.0 / a;
        }
        __syncthreads();
        if (tid == 0) {
            const double floor_w = 10.0 * 2.220446049250313e-16;
            double W = 0.0, b = 0.0;
            for (int g = 0; g < m; ++g) if (gw[g] >= floor_w) W += gw[g];
            for (int g = 0; g < m; ++g) if (gw[g] >= floor_w) b += gb[g] * (gw[g] / W);
            sh_b = b;
        }
        __syncthreads();
        const double b = sh_b;
        double kp = 0.0;
        for (int j = tid; j < nt; j += PS_THREADS) kp += log1p(-b * ty[j]);
        kp = ps_reduce(kp, red, PsSum()) / (double)nt;
        const double sigma = -kp / b;
        khat = gpd_k_prior(kp, nt);
        if (isfinite(khat))
            for (int j = tid; j < nt; j += PS_THREADS) {
                double t = log(gpd_inv(((double)j + 0.5) / (double)nt, khat, sigma) + ec);
                if (t > 0.0) t = 0.0;
                tv[j] = t;
            }
        __syncthreads();
    }
    // log weights lw = x' - logsumexp(x'), then elpd = logsumexp(lw + ll): the body draws (x <= cutoff), then the tail
    double xm = -HUGE_VAL;
    for (int s = tid; s < S; s += PS_THREADS) { const double x = mn - v[s]; if (!(x > cutoff)) xm = fmax(xm, x); }
    for (int j = tid; j < nt; j += PS_THREADS) xm = fmax(xm, tv[j]);
    xm = ps_reduce(xm, red, PsMax());
    double se = 0.0;
    for (int s = tid; s < S; s += PS_THREADS) { const double x = mn - v[s]; if (!(x > cutoff)) se += exp(x - xm); }
    for (int j = tid; j < nt; j += PS_THREADS) se += exp(tv[j] - xm);
    const double lse = xm + log(ps_reduce(se, red, PsSum()));
    double tm = -HUGE_VAL;
    for (int s = tid; s < S; s += PS_THREADS) { const double x = mn - v[s]; if (!(x > cutoff)) tm = fmax(tm, (x - lse) + v[s]); }
    for (int j = tid; j < nt; j += PS_THREADS) tm = fmax(tm, (tv[j] - lse) + v[ti[j]]);
    tm = ps_reduce(tm, red, PsMax());
    double st = 0.0;
    for (int s = tid; s < S; s += PS_THREADS) { const double x = mn - v[s]; if (!(x > cutoff)) st += exp(((x - lse) + v[s]) - tm); }
    for (int j = tid; j < nt; j += PS_THREADS) st += exp(((tv[j] - lse) + v[ti[j]]) - tm);
    st = ps_reduce(st, red, PsSum());
    if (tid == 0) {
        elpd_out[obs] = tm + log(st);
        k_out[obs] = khat;
        lppd_out[obs] = mx + log(e) - log((double)S);
        pw_out[obs] = q / (double)(S - 1);
    }
}

int launch_psis(const double *ll, int64_t n_draws, int64_t n_obs, double *elpd, double *khat, double *lppd, double *p_waic)
{
    if (n_obs <= 0) return 0;
    if (n_draws < 2 || n_draws > PSIS_MAX_DRAWS) { g_be_err = "k_psis takes 2 .. 16384 draws"; return -1; }
    const size_t smem = sizeof(double) * (size_t)n_draws;
    CU(cudaFuncSetAttribute(k_psis, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(double) * PSIS_MAX_DRAWS)));
    k_psis<<<(unsigned)n_obs, PS_THREADS, smem, stream()>>>(ll, (int)n_draws, elpd, khat, lppd, p_waic);
    LAUNCHED("k_psis");
    return 0;
}

// ------------------------------------------------------------------------------------------------
// migration (migration.jl:11-116)
// ------------------------------------------------------------------------------------------------
// select_particle (migration.jl:89-95): p ~ exp(-w)/sum(exp(-w)); NaN => findmin(w), no draw
__device__ int select_particle_block(const double *w, int Np, double u, double *th /*smem Np*/)
{
    __shared__ double s_tot;
    __shared__ int s_res;
    for (int i = threadIdx.x; i < Np; i += blockDim.x) th[i] = exp(-w[i]);
    __syncthreads();
    if (threadIdx.x == 0) { ksum_t k = { 0.0, 0.0 }; for (int i = 0; i < Np; ++i) kadd(k, th[i]); s_tot = kval(k); }
    __syncthreads();
    bool bad = false;
    for (int i = threadIdx.x; i < Np; i += blockDim.x) { const double v = th[i] / s_tot; th[i] = v; bad |= (v != v); }
    const int any_bad = __syncthreads_or(bad ? 1 : 0);
    if (threadIdx.x == 0) {
        int r = 0;
        if (any_bad) {
            for (int i = 0; i < Np; ++i) { if (w[i] != w[i]) { r = i; break; } if (w[i] < w[r]) r = i; }
        } else {
            ksum_t k = { 0.0, 0.0 };
            for (int i = 0; i < Np; ++i) kadd(k, th[i]);
            const double t = u * kval(k);
            double cw = th[0];
            while (cw < t && r < Np - 1) { ++r; cw += th[r]; }
        }
        s_res = r;
    }
    __syncthreads();
    return s_res;
}

// select_base (crossover.jl:282-289), single block; used by demcmc_op_select
__device__ int select_base_block(const double *w, int Np, double u, double *th)
{
    __shared__ double s_tot;
    __shared__ int s_res;
    for (int i = threadIdx.x; i < Np; i += blockDim.x) th[i] = exp(w[i]);
    __syncthreads();
    if (threadIdx.x == 0) { ksum_t k = { 0.0, 0.0 }; for (int i = 0; i < Np; ++i) kadd(k, th[i]); s_tot = kval(k); }
    __syncthreads();
    bool bad = false;
    for (int i = threadIdx.x; i < Np; i += blockDim.x) { const double v = th[i] / s_tot; th[i] = v; bad |= (v != v); }
    const int any_bad = __syncthreads_or(bad ? 1 : 0);
    if (threadIdx.x == 0) {
        const double *src = any_bad ? w : th;
        ksum_t k = { 0.0, 0.0 };
        for (int i = 0; i < Np; ++i) kadd(k, src[i]);
        const double t = u * kval(k);
        int r = 0;
        double cw = src[0];
        while (cw < t && r < Np - 1) { ++r; cw += src[r]; }
        s_res = r;
    }
    __syncthreads();
    return s_res;
}

__global__ void __launch_bounds__(128) k_mig_pick(ConfigDev cfg, MigArgs a, const double *w, int32_t *picks)
{
    extern __shared__ double th[];
    const int i = blockIdx.x, gl = a.groups[i] - cfg.group_begin;
    if (gl < 0 || gl >= cfg.G_local) { if (threadIdx.x == 0) picks[i] = -1; return; }
    const int r = select_particle_block(w + (size_t)gl * cfg.Np, cfg.Np, a.u_pick[i], th);
    if (threadIdx.x == 0) picks[i] = r;
}

// The whole Particle object migrates (theta, weight, id and its accept/lp history): the staging row
// is {theta[d], weight, id, accept flag of the row being edited}
__global__ void __launch_bounds__(128) k_mig_gather(ConfigDev cfg, MigArgs a, const int32_t *picks, const double *theta,
                                                    const double *w, const int32_t *id, const uint8_t *acc, double *stage)
{
    const int i = blockIdx.x, gl = a.groups[i] - cfg.group_begin;
    if (gl < 0 || gl >= cfg.G_local) return;
    const size_t p = (size_t)gl * cfg.Np + picks[i];
    double *row = stage + (size_t)i * (cfg.d + 3);
    for (int k = threadIdx.x; k < cfg.d; k += blockDim.x) row[k] = theta[p * cfg.d + k];
    if (threadIdx.x == 0) { row[cfg.d] = w[p]; row[cfg.d + 1] = (double)id[p]; row[cfg.d + 2] = (double)acc[p]; }
}

// shift_particles! (migration.jl:109-116): position i receives the particle picked at position i-1
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long *p)
{
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];\n" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__global__ void __launch_bounds__(128) k_mig_scatter(ConfigDev cfg, MigArgs a, const int32_t *picks, const double *stage,
                                                     double *theta, double *w, int32_t *id, uint8_t *acc, int32_t *pos,
                                                     Mbox mbox, int rank, int slot, unsigned long long tag)
{
    const int i = blockIdx.x, gl = a.groups[i] - cfg.group_begin;
    if (gl < 0 || gl >= cfg.G_local) return;
    const size_t p = (size_t)gl * cfg.Np + picks[i];
    const int r = (i + a.n - 1) % a.n;
    const double *row = stage + (size_t)r * (cfg.d + 3);
    if (mbox.rows && a.src_rank[i] != rank) {
        // the row was produced on another rank: it arrives in this rank's mailbox (k_mig_push over NVLink)
        const size_t cell = (size_t)slot * mbox.max_rows + r;
        if (threadIdx.x == 0) {
            const unsigned long long t0 = gtime();
            while (ld_acquire_sys_u64(mbox.flags + cell) != tag) {
                __nanosleep(100);
                if (gtime() - t0 > 30000000000ull) __trap();      // a peer that never arrives: trap, do not hang the device
            }
        }
        __syncthreads();
        row = mbox.rows + cell * mbox.row_len;
    }
    for (int k = threadIdx.x; k < cfg.d; k += blockDim.x) theta[p * cfg.d + k] = __ldcv(row + k);
    if (threadIdx.x == 0) {
        const double rw = __ldcv(row + cfg.d), rid = __ldcv(row + cfg.d + 1), ra = __ldcv(row + cfg.d + 2);
        w[p] = rw; id[p] = (int32_t)rid; acc[p] = (uint8_t)ra;
        if (pos) pos[(int32_t)rid - cfg.group_begin * cfg.Np] = (int32_t)p;
    }
}

// rows produced here and consumed on another rank: store them into the consumer's mailbox, then publish the tag
__global__ void __launch_bounds__(128) k_mig_push(ConfigDev cfg, MigArgs a, const double *stage, PeerTable peers, Mbox geom,
                                                  int rank, int slot, unsigned long long tag)
{
    const int i = blockIdx.x;
    if (a.src_rank[i] != rank || a.dst_rank[i] == rank) return;
    const int r = (i + a.n - 1) % a.n, dst = a.dst_rank[i];
    const size_t cell = (size_t)slot * geom.max_rows + r;
    const double *row = stage + (size_t)r * (cfg.d + 3);
    double *out = peers.rows[dst] + cell * geom.row_len;
    for (int k = threadIdx.x; k < cfg.d + 3; k += blockDim.x) out[k] = row[k];
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) asm volatile("st.release.sys.global.u64 [%0], %1;\n" ::"l"(peers.flags[dst] + cell), "l"(tag) : "memory");
}

int launch_mig_pick(const ConfigDev &cfg, const MigArgs &a, const double *w, int32_t *picks)
{
    k_mig_pick<<<a.n, 128, sizeof(double) * cfg.Np, stream()>>>(cfg, a, w, picks);
    LAUNCHED("k_mig_pick");
    return 0;
}
int launch_mig_gather(const ConfigDev &cfg, const MigArgs &a, const int32_t *picks, const double *theta, const double *w,
                      const int32_t *id, const uint8_t *acc, double *stage)
{
    k_mig_gather<<<a.n, 128, 0, stream()>>>(cfg, a, picks, theta, w, id, acc, stage);
    LAUNCHED("k_mig_gather");
    return 0;
}
int launch_mig_scatter(const ConfigDev &cfg, const MigArgs &a, const int32_t *picks, const double *stage, double *theta,
                       double *w, int32_t *id, uint8_t *acc, int32_t *pos, const Mbox *mbox, int rank, int slot, unsigned long long tag)
{
    Mbox none = { nullptr, nullptr, 0, 0, 0 };
    k_mig_scatter<<<a.n, 128, 0, stream()>>>(cfg, a, picks, stage, theta, w, id, acc, pos, mbox ? *mbox : none, rank, slot, tag);
    LAUNCHED("k_mig_scatter");
    return 0;
}
int launch_mig_push(const ConfigDev &cfg, const MigArgs &a, const double *stage, const PeerTable &peers, const Mbox &geom,
                    int rank, int slot, unsigned long long tag)
{
    k_mig_push<<<a.n, 128, 0, stream()>>>(cfg, a, stage, peers, geom, rank, slot, tag);
    LAUNCHED("k_mig_push");
    return 0;
}
// The mailbox is plain cudaMalloc memory: stream-ordered pool memory cannot be exported with cudaIpcGetMemHandle
int mbox_create(int depth, int max_rows, int row_len, Mbox *out)
{
    out->depth = depth; out->max_rows = max_rows; out->row_len = row_len; out->rows = nullptr; out->flags = nullptr;
    const size_t cells = (size_t)depth * max_rows;
    CU(cudaMalloc(&out->rows, sizeof(double) * cells * row_len));
    CU(cudaMalloc(&out->flags, sizeof(unsigned long long) * cells));
    CU(cudaMemset(out->flags, 0, sizeof(unsigned long long) * cells));
    CU(cudaDeviceSynchronize());
    return 0;
}
void mbox_destroy(Mbox *m) { if (m->rows) cudaFree(m->rows); if (m->flags) cudaFree(m->flags); m->rows = nullptr; m->flags = nullptr; }
int mbox_export(const Mbox &m, uint8_t handle[128])
{
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "two IPC handles fill the 128-byte blob");
    cudaIpcMemHandle_t hr, hf;
    CU(cudaIpcGetMemHandle(&hr, m.rows));
    CU(cudaIpcGetMemHandle(&hf, m.flags));
    memcpy(handle, &hr, 64); memcpy(handle + 64, &hf, 64);
    return 0;
}
int mbox_open(const uint8_t handle[128], Mbox *peer)
{
    cudaIpcMemHandle_t hr, hf;
    memcpy(&hr, handle, 64); memcpy(&hf, handle + 64, 64);
    CU(cudaIpcOpenMemHandle((void **)&peer->rows, hr, cudaIpcMemLazyEnablePeerAccess));
    CU(cudaIpcOpenMemHandle((void **)&peer->flags, hf, cudaIpcMemLazyEnablePeerAccess));
    return 0;
}
void mbox_close(Mbox *peer) { if (peer->rows) cudaIpcCloseMemHandle(peer->rows); if (peer->flags) cudaIpcCloseMemHandle(peer->flags); peer->rows = nullptr; peer->flags = nullptr; }
int enable_peer_access(int dev, int peer_dev)
{
    if (dev == peer_dev) return 0;
    int can = 0;
    CU(cudaDeviceCanAccessPeer(&can, dev, peer_dev));
    if (!can) { g_be_err = "no peer access between the two devices"; return -1; }
    int keep = 0;
    CU(cudaGetDevice(&keep));
    CU(cudaSetDevice(dev));
    cudaError_t e = cudaDeviceEnablePeerAccess(peer_dev, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) { (void)cudaGetLastError(); e = cudaSuccess; }
    cudaSetDevice(keep);
    if (e != cudaSuccess) return cu_fail(e, "cudaDeviceEnablePeerAccess");
    // device memory here comes from the stream-ordered pool (dmalloc), which peer access does not cover by itself:
    // `dev` must be granted access to peer_dev's pool as well
    cudaMemPool_t pool;
    CU(cudaDeviceGetDefaultMemPool(&pool, peer_dev));
    cudaMemAccessDesc desc = {};
    desc.location.type = cudaMemLocationTypeDevice; desc.location.id = dev; desc.flags = cudaMemAccessFlagsProtReadWrite;
    CU(cudaMemPoolSetAccess(pool, &desc, 1));
    return 0;
}

// ------------------------------------------------------------------------------------------------
// history: rows by slot -> samples[P][d][n_rows] / lp[P][n_rows] / accept[P][n_rows] by particle id
// (the memory order of Julia's Array{T,3}(n_rows, d, P), utilities.jl:34).  Lanes run along rows so
// the writes coalesce.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_history(const double *rt, const double *rw, const uint8_t *ra, const int32_t *rid,
                                                 int64_t n_rows_dev, int64_t row0, int64_t n_rows_out, int P, int d, int id_base,
                                                 double *samples, double *lp, uint8_t *accept, int P_ids)
{
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int slot = blockIdx.y;
    if (r >= n_rows_dev) return;
    const int id = rid[r * P + slot] - id_base;
    if (id < 0 || id >= P_ids) return;
    const int64_t ro = row0 + r;
    if (samples) for (int k = 0; k < d; ++k) samples[((int64_t)id * d + k) * n_rows_out + ro] = rt[(r * P + slot) * d + k];
    if (lp) lp[(int64_t)id * n_rows_out + ro] = rw[r * P + slot];
    if (accept) accept[(int64_t)id * n_rows_out + ro] = ra[r * P + slot];
}

int launch_history_by_id(const double *rows_theta, const double *rows_w, const uint8_t *rows_acc, const int32_t *rows_id,
                         int64_t n_rows_dev, int64_t row0, int64_t n_rows_out, int32_t P, int32_t d, int32_t id_base,
                         double *samples, double *lp, uint8_t *accept, int32_t P_ids)
{
    dim3 grid((unsigned)((n_rows_dev + 255) / 256), (unsigned)P);
    k_history<<<grid, 256, 0, stream()>>>(rows_theta, rows_w, rows_acc, rows_id, n_rows_dev, row0, n_rows_out, P, d, id_base, samples, lp, accept, P_ids > 0 ? P_ids : P);
    LAUNCHED("k_history");
    return 0;
}

// bundle_samples (main.jl:222-250) on the device: chains[c][k][row] for rows [row0, row0+n_rows) of
// the history; parameter columns k < d of chain c are the draws of particle id c, the columns
// "acceptance" (d) and "lp" (d+1) belong to the particle sitting at final position c
__global__ void __launch_bounds__(256) k_chain_pos(const int32_t *final_id, int P, int id_base, int32_t *pos_of_id, int P_ids, int pos_base)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= P) return;
    const int id = final_id[c] - id_base;
    if (id >= 0 && id < P_ids) pos_of_id[id] = pos_base + c;
}
__global__ void __launch_bounds__(256) k_chains(const double *rt, const double *rw, const uint8_t *ra, const int32_t *rid,
                                                const int32_t *pos_of_id, int64_t row0, int64_t n_rows, int P, int d, int id_base, double *out, int P_ids)
{
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int slot = blockIdx.y;
    if (r >= n_rows) return;
    const int64_t row = row0 + r;
    const int id = rid[row * P + slot] - id_base;
    if (id < 0 || id >= P_ids) return;
    const double *src = rt + (row * P + slot) * d;
    double *dst = out + (int64_t)id * (d + 2) * n_rows + r;
    for (int k = 0; k < d; ++k) dst[(int64_t)k * n_rows] = src[k];
    double *dq = out + (int64_t)pos_of_id[id] * (d + 2) * n_rows + r;
    dq[(int64_t)d * n_rows] = (double)ra[row * P + slot];
    dq[(int64_t)(d + 1) * n_rows] = rw[row * P + slot];
}

int launch_chains(const double *rows_theta, const double *rows_w, const uint8_t *rows_acc, const int32_t *rows_id,
                  const int32_t *final_id, int32_t *pos_scratch, int64_t row0, int64_t n_rows, int32_t P, int32_t d, int32_t id_base, double *out,
                  int32_t P_ids, int32_t pos_base, int phase)
{
    if (P_ids <= 0) P_ids = P;
    if (phase & 1) {
        k_chain_pos<<<(P + 255) / 256, 256, 0, stream()>>>(final_id, P, id_base, pos_scratch, P_ids, pos_base);
        LAUNCHED("k_chain_pos");
    }
    if (n_rows <= 0 || !(phase & 2)) return 0;
    dim3 grid((unsigned)((n_rows + 255) / 256), (unsigned)P);
    k_chains<<<grid, 256, 0, stream()>>>(rows_theta, rows_w, rows_acc, rows_id, pos_scratch, row0, n_rows, P, d, id_base, out, P_ids);
    LAUNCHED("k_chains");
    return 0;
}

// ------------------------------------------------------------------------------------------------
// streaming moments of the history: Welford per thread over the vectors of its block, Chan's merge
// of the per-block partials in block order (deterministic; lanes run along the parameters, so the
// reads coalesce).  Both work on x - x[0] (the first vector): the partial means are then of the size of
// the spread, and the differences of them in the merge do not cancel for a parameter at a large offset
// ------------------------------------------------------------------------------------------------
constexpr int MOM_BLOCKS = 592, MOM_THREADS = 128;
__global__ void __launch_bounds__(MOM_THREADS) k_moments_partial(const double *x, int64_t n, int d, double *pmean, double *pm2)
{
    for (int k = threadIdx.x; k < d; k += MOM_THREADS) {
        double mean = 0.0, m2 = 0.0, cnt = 0.0;
        const double shift = x[k];
        for (int64_t r = blockIdx.x; r < n; r += MOM_BLOCKS) {
            const double v = x[r * d + k] - shift;
            cnt += 1.0;
            const double dl = v - mean;
            mean += dl / cnt;
            m2 += dl * (v - mean);
        }
        pmean[(size_t)blockIdx.x * d + k] = mean;
        pm2[(size_t)blockIdx.x * d + k] = m2;
    }
}
__global__ void __launch_bounds__(MOM_THREADS) k_moments_merge(const double *x, const double *pmean, const double *pm2, int64_t n, int d, double *mean, double *m2)
{
    const int k = blockIdx.x * MOM_THREADS + threadIdx.x;
    if (k >= d) return;
    double ca = 0.0, ma = 0.0, sa = 0.0;
    for (int b = 0; b < MOM_BLOCKS; ++b) {
        const double cb = (double)((n - b + MOM_BLOCKS - 1) / MOM_BLOCKS);       // vectors block b saw
        if (cb <= 0.0) break;
        const double mb = pmean[(size_t)b * d + k], sb = pm2[(size_t)b * d + k];
        const double dl = mb - ma, c = ca + cb;
        ma += dl * (cb / c);
        sa += sb + dl * dl * (ca * cb / c);
        ca = c;
    }
    mean[k] = x[k] + ma; m2[k] = sa;
}
int launch_moments(const double *x, int64_t n, int32_t d, double *mean, double *m2)
{
    double *part = (double *)dmalloc(sizeof(double) * 2 * (size_t)MOM_BLOCKS * d);
    if (!part) return -1;
    k_moments_partial<<<MOM_BLOCKS, MOM_THREADS, 0, stream()>>>(x, n, d, part, part + (size_t)MOM_BLOCKS * d);
    LAUNCHED("k_moments_partial");
    k_moments_merge<<<(d + MOM_THREADS - 1) / MOM_THREADS, MOM_THREADS, 0, stream()>>>(x, part, part + (size_t)MOM_BLOCKS * d, n, d, mean, m2);
    LAUNCHED("k_moments_merge");
    dfree(part);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// convergence diagnostics of the stored history, on the device (backend.h: launch_diag_aggregates)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_diag_pos(const int32_t *rid, int64_t row0, int64_t n_rows, int P, int id_base, int P_ids, int pos_base, int32_t *pos)
{
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n_rows * P) return;
    const int64_t r = i / P;
    const int id = rid[(row0 + r) * P + (i - r * P)] - id_base;
    if (id >= 0 && id < P_ids) pos[r * P_ids + id] = pos_base + (int32_t)(i - r * P);
}
// one block per (parameter k, group of chains): each split chain is gathered into shared memory (its draws sit at a
// different position of every stored row: ids migrate), then thread t accumulates the lags t, t + 256, ...; the
// block's chains are summed in order, the groups by k_diag_merge in order: deterministic.
// Every draw is taken less c_k, the draw of id 0 at row0 (the same value in every block and shard): the chain means and
// the sums of them and of their squares are then of the size of the spread, not of the location, so the between-chain
// variance diag_finish forms from them does not cancel for a parameter at a large offset (agg[1] and agg[2] are of the
// shifted means; the variances and autocovariances do not depend on the shift).
constexpr int DG_THREADS = 256, DG_GROUPS = 32, DG_MAX_LAG = 4096 /* lags per launch: 16 accumulators per thread */, DG_MAX_NH = 24576 /* 192 KB of shared memory */;
__global__ void __launch_bounds__(DG_THREADS) k_diag_partial(DiagShards sh, const int32_t *pos, int64_t row0, int64_t n_rows, int P, int d,
                                                             int lag0, int n_lag, double *part /* [d][DG_GROUPS][3 + n_lag]: lags lag0 .. lag0 + n_lag - 1 */)
{
    extern __shared__ double xs[];                                // nh draws of one split chain
    __shared__ double red[DG_THREADS / 32 + 1];
    const int k = blockIdx.x, grp = blockIdx.y, tid = threadIdx.x;
    const int nh = (int)(n_rows / 2);
    const int n_chain = 2 * P;
    const int c0 = (int)((int64_t)grp * n_chain / DG_GROUPS), c1 = (int)((int64_t)(grp + 1) * n_chain / DG_GROUPS);
    double *out = part + ((size_t)k * DG_GROUPS + grp) * (3 + n_lag);
    double s_cv = 0.0, s_m = 0.0, s_m2 = 0.0;
    constexpr int LPT = (DG_MAX_LAG + DG_THREADS - 1) / DG_THREADS; // lags per thread
    double acov[LPT];
#pragma unroll
    for (int j = 0; j < LPT; ++j) acov[j] = 0.0;
    const int q0 = pos[0], shard0 = q0 / sh.P_local;
    const double shift = sh.theta[shard0][(row0 * sh.P_local + (q0 - shard0 * sh.P_local)) * d + k];
    for (int c = c0; c < c1; ++c) {
        const int id = c >> 1;
        const int64_t r0 = (c & 1) ? n_rows - nh : 0;             // second half: the LAST nh draws
        double s = 0.0;
        for (int i = tid; i < nh; i += DG_THREADS) {
            const int64_t r = r0 + i;
            const int q = pos[r * P + id], shard = q / sh.P_local;
            const double v = sh.theta[shard][((row0 + r) * sh.P_local + (q - shard * sh.P_local)) * d + k] - shift;
            xs[i] = v; s += v;
        }
        s = warp_sum(s);
        __syncthreads();
        if ((tid & 31) == 0) red[tid >> 5] = s;
        __syncthreads();
        double mean = 0.0;
        for (int w = 0; w < DG_THREADS / 32; ++w) mean += red[w];
        mean /= (double)nh;
        __syncthreads();
        for (int i = tid; i < nh; i += DG_THREADS) xs[i] -= mean;
        __syncthreads();
#pragma unroll
        for (int j = 0; j < LPT; ++j) {
            const int tl = tid + j * DG_THREADS, t = lag0 + tl;
            if (tl < n_lag) {
                double a = 0.0;
                for (int i = 0; i + t < nh; ++i) a += xs[i] * xs[i + t];
                a /= (double)nh;
                acov[j] += a;
                if (t == 0) { s_cv += a * (double)nh / (double)(nh - 1); s_m += mean; s_m2 += mean * mean; }
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int j = 0; j < LPT; ++j) { const int t = tid + j * DG_THREADS; if (t < n_lag) out[3 + t] = acov[j]; }
    if (tid == 0) { out[0] = s_cv; out[1] = s_m; out[2] = s_m2; }
}
__global__ void __launch_bounds__(256) k_diag_merge(const double *part, int d, int n_lag, double *agg)
{
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= (int64_t)d * (3 + n_lag)) return;
    const int k = (int)(i / (3 + n_lag)), j = (int)(i - (int64_t)k * (3 + n_lag));
    double s = 0.0;
    for (int g = 0; g < DG_GROUPS; ++g) s += part[((size_t)k * DG_GROUPS + g) * (3 + n_lag) + j];
    agg[i] = s;
}
int launch_diag_pos(const int32_t *rows_id, int64_t row0, int64_t n_rows, int32_t P_local, int32_t id_base, int32_t P_ids, int32_t pos_base, int32_t *pos)
{
    k_diag_pos<<<(unsigned)((n_rows * P_local + 255) / 256), 256, 0, stream()>>>(rows_id, row0, n_rows, P_local, id_base, P_ids, pos_base, pos);
    LAUNCHED("k_diag_pos");
    return 0;
}
int diag_max_half() { return DG_MAX_NH; }
int diag_max_lags() { return DG_MAX_LAG; }
int launch_diag_aggregates(const DiagShards &sh, const int32_t *pos, int64_t row0, int64_t n_rows, int32_t P_ids, int32_t d, int32_t lag0, int32_t n_lag, double *agg)
{
    const int64_t nh = n_rows / 2;
    if (nh < 2 || nh > DG_MAX_NH || lag0 < 0 || n_lag < 1 || n_lag > DG_MAX_LAG || lag0 + n_lag > nh) { g_be_err = "diagnostics need 4 <= n_rows <= 49152 stored rows and at most 4096 lags per launch"; return -1; }
    if (sizeof(double) * nh > 48 * 1024) {
        static bool attr_set[64] = {};
        if (!attr_set[g_dev & 63]) {
            if (cudaFuncSetAttribute(k_diag_partial, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(double) * DG_MAX_NH)) != cudaSuccess) { g_be_err = "k_diag_partial: shared-memory opt-in refused"; return -1; }
            attr_set[g_dev & 63] = true;
        }
    }
    double *part = (double *)dmalloc(sizeof(double) * (size_t)d * DG_GROUPS * (3 + n_lag));
    if (!part) return -1;
    k_diag_partial<<<dim3(d, DG_GROUPS), DG_THREADS, sizeof(double) * nh, stream()>>>(sh, pos, row0, n_rows, P_ids, d, lag0, n_lag, part);
    LAUNCHED("k_diag_partial");
    k_diag_merge<<<(unsigned)(((int64_t)d * (3 + n_lag) + 255) / 256), 256, 0, stream()>>>(part, d, n_lag, agg);
    LAUNCHED("k_diag_merge");
    dfree(part);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// power posteriors (demcmc_power_posterior): the per-slice partials of the stored untempered log-likelihoods
// ------------------------------------------------------------------------------------------------
constexpr int PP_THREADS = 256;
// sum and max over the block in a fixed order (lanes by the xor tree, then the warps in order), the same value to every thread
__device__ __forceinline__ void pp_block_reduce(double &s, double &mx, double *red)
{
    for (int o = 16; o > 0; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o)); }
    __syncthreads();
    if ((threadIdx.x & 31) == 0) { red[2 * (threadIdx.x >> 5)] = s; red[2 * (threadIdx.x >> 5) + 1] = mx; }
    __syncthreads();
    s = 0.0; mx = -inf();
    for (int w = 0; w < PP_THREADS / 32; ++w) { s += red[2 * w]; mx = fmax(mx, red[2 * w + 1]); }
}
// one block per (slice, local group): rows [row0 + slice * PP_ROWS, ...) of the group's Np positions.  Two passes over the
// slice: count, sum and max; then the squared deviations from the slice mean and the exponentials shifted by the slice max.
// (Without migration a particle never leaves its group, so the positions of a group hold the group's ids at every row.)
__global__ void __launch_bounds__(PP_THREADS) k_power_posterior(const double *ll, int64_t row0, int64_t n_rows, int P, int Np,
                                                                const PPDelta delta, double *part /* [G_local][n_slices][PP_OUT] */)
{
    __shared__ double red[2 * (PP_THREADS / 32)];
    const int s = blockIdx.x, g = blockIdx.y, n_slices = gridDim.x;
    const int64_t r0 = row0 + (int64_t)s * PP_ROWS, nr = min((int64_t)PP_ROWS, row0 + n_rows - r0), n = nr * Np;
    const double dl = delta.v[g];
    auto at = [&](int64_t e) { const int64_t r = e / Np; return ll[(r0 + r) * P + (size_t)g * Np + (e - r * Np)]; };
    double sum = 0.0, mx = -inf();
    for (int64_t e = threadIdx.x; e < n; e += PP_THREADS) { const double v = at(e); sum += v; mx = fmax(mx, v); }
    pp_block_reduce(sum, mx, red);
    const double mean = sum / (double)n;
    double m2 = 0.0, e1 = 0.0, e2 = 0.0;
    for (int64_t e = threadIdx.x; e < n; e += PP_THREADS) {
        const double v = at(e), dv = v - mean, x = exp(dl * (v - mx));
        m2 += dv * dv; e1 += x; e2 += x * x;
    }
    double unused = -inf();
    pp_block_reduce(m2, unused, red);
    unused = -inf();
    pp_block_reduce(e1, unused, red);
    unused = -inf();
    pp_block_reduce(e2, unused, red);
    if (threadIdx.x == 0) {
        double *o = part + ((size_t)g * n_slices + s) * PP_OUT;
        o[0] = (double)n; o[1] = mean; o[2] = m2; o[3] = mx; o[4] = e1; o[5] = e2;
    }
}
__global__ void __launch_bounds__(256) k_temper_weights(ConfigDev cfg, const double *prior, const double *ll, int64_t n, double *w)
{
    const int64_t p = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (p >= n) return;
    const double pr = prior[p];
    w[p] = pr == -inf() ? -inf() : add(pr, tempered_ll(cfg, cfg.group_begin + (int)(p / cfg.Np), ll[p]));
}
int launch_temper_weights(const ConfigDev &cfg, const double *prior, const double *ll, int64_t n, double *w)
{
    if (n <= 0) return 0;
    k_temper_weights<<<(unsigned)((n + 255) / 256), 256, 0, stream()>>>(cfg, prior, ll, n, w);
    LAUNCHED("k_temper_weights");
    return 0;
}
int launch_power_posterior(const double *ll_rows, int64_t row0, int64_t n_rows, int32_t P_local, int32_t Np, int32_t G_local,
                           const PPDelta &delta, double *part)
{
    const int64_t n_slices = (n_rows + PP_ROWS - 1) / PP_ROWS;
    if (n_rows < 1 || G_local < 1 || G_local > MAX_MIG || n_slices > INT32_MAX) { g_be_err = "power posterior: bad row range or group count"; return -1; }
    k_power_posterior<<<dim3((unsigned)n_slices, (unsigned)G_local), PP_THREADS, 0, stream()>>>(ll_rows, row0, n_rows, P_local, Np, delta, part);
    LAUNCHED("k_power_posterior");
    return 0;
}

// ------------------------------------------------------------------------------------------------
// particle algebra ops (single warp)
// ------------------------------------------------------------------------------------------------
__global__ void k_op_project(const double *p1, const double *p2, int d, double *out)
{
    const int lane = threadIdx.x;
    double v1 = 0.0, v2 = 0.0;
    for (int k = lane; k < d; k += 32) { v1 = add(v1, mul(p1[k], p2[k])); v2 = add(v2, mul(p2[k], p2[k])); }
    v1 = warp_sum(v1); v2 = warp_sum(v2);
    const double r = v1 / v2;
    for (int k = lane; k < d; k += 32) out[k] = mul(p2[k], r);
}
__global__ void k_op_snooker(const double *pt, const double *pz, const double *pm, const double *pn, double g,
                             const double *b, int d, double *out, double *log_adj)
{
    const int lane = threadIdx.x;
    double v1m = 0.0, v1n = 0.0, v2 = 0.0;
    for (int k = lane; k < d; k += 32) {
        const double pd = sub(pt[k], pz[k]);
        v1m = add(v1m, mul(pm[k], pd)); v1n = add(v1n, mul(pn[k], pd)); v2 = add(v2, mul(pd, pd));
    }
    v1m = warp_sum(v1m); v1n = warp_sum(v1n); v2 = warp_sum(v2);
    const double r1 = v1m / v2, r2 = v1n / v2;
    double sq1 = 0.0, sq2 = 0.0;
    for (int k = lane; k < d; k += 32) {
        const double v = snooker_elem(pt[k], pz[k], r1, r2, g, b[k]);
        out[k] = v;
        const double a = sub(v, pz[k]), c = sub(pt[k], pz[k]);
        sq1 = add(sq1, mul(a, a)); sq2 = add(sq2, mul(c, c));
    }
    sq1 = warp_sum(sq1); sq2 = warp_sum(sq2);
    if (lane == 0) *log_adj = adjust_loglike(sq1, sq2, d);
}
__global__ void k_op_de(const double *pt, const double *pm, const double *pn, const double *pb, double g1, double g2,
                        const double *b, int d, double *out)
{
    for (int k = threadIdx.x; k < d; k += 32) out[k] = de_elem(pt[k], pm[k], pn[k], pb ? pb[k] : pt[k], g1, g2, pb != nullptr, b[k]);
}
__global__ void k_op_reset(const double *prop, const double *pt, const uint8_t *mask, int d, double *out)
{
    for (int k = threadIdx.x; k < d; k += 32) out[k] = mask[k] ? prop[k] : pt[k];
}
__global__ void k_op_accept(const double *wp, const double *wc, const double *adj, const double *u, int n, uint8_t *out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = accept(wp[i], wc[i], adj[i], u[i]) ? 1 : 0;
}
__global__ void __launch_bounds__(128) k_op_select(const double *w, int n, double u, int32_t *base_idx, int32_t *mig_idx)
{
    extern __shared__ double th[];
    const int b = select_base_block(w, n, u, th);
    __syncthreads();
    const int q = select_particle_block(w, n, u, th);
    if (threadIdx.x == 0) { *base_idx = b; *mig_idx = q; }
}

int launch_op_project(const double *p1, const double *p2, int d, double *out) { k_op_project<<<1, 32, 0, stream()>>>(p1, p2, d, out); LAUNCHED("k_op_project"); return 0; }
int launch_op_snooker(const double *pt, const double *pz, const double *pm, const double *pn, double g, const double *b, int d, double *out, double *log_adj)
{ k_op_snooker<<<1, 32, 0, stream()>>>(pt, pz, pm, pn, g, b, d, out, log_adj); LAUNCHED("k_op_snooker"); return 0; }
int launch_op_de(const double *pt, const double *pm, const double *pn, const double *pb, double g1, double g2, const double *b, int d, double *out)
{ k_op_de<<<1, 32, 0, stream()>>>(pt, pm, pn, pb, g1, g2, b, d, out); LAUNCHED("k_op_de"); return 0; }
int launch_op_reset(const double *prop, const double *pt, const uint8_t *mask, int d, double *out) { k_op_reset<<<1, 32, 0, stream()>>>(prop, pt, mask, d, out); LAUNCHED("k_op_reset"); return 0; }
int launch_op_accept(const double *wp, const double *wc, const double *adj, const double *u, int n, uint8_t *out)
{ k_op_accept<<<(n + 127) / 128, 128, 0, stream()>>>(wp, wc, adj, u, n, out); LAUNCHED("k_op_accept"); return 0; }
int launch_op_select(const double *w, int n, double u, int32_t *base_idx, int32_t *mig_idx)
{ k_op_select<<<1, 128, sizeof(double) * n, stream()>>>(w, n, u, base_idx, mig_idx); LAUNCHED("k_op_select"); return 0; }

// ------------------------------------------------------------------------------------------------
// roofline probes
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_dfma_peak(double *out, int iters, double a, double b)
{
    double r[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) r[i] = (double)(threadIdx.x + i);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 16; ++i) r[i] = fma(r[i], a, b);
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += r[i];
    if (s == 123.456) out[0] = s;
}

// the fp64 tensor path: 8 independent DMMA m8n8k4 chains per warp
__global__ void __launch_bounds__(256) k_dmma_peak(double *out, int iters, double a, double b)
{
    double c[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) c[i] = 0.0;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 8; ++i) dmma884(c[2 * i], c[2 * i + 1], a, b);
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += c[i];
    if (s == 123.456) out[0] = s;
}

// DFMA loop and DMMA loop, best of 5 timed repetitions each, TFLOP/s
int fp64_peaks(double *dfma_tflops, double *dmma_tflops)
{
    int sms = 0;
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, g_dev));
    double *out = (double *)dmalloc(8);
    if (!out) return -1;
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
    const int blocks = sms * 8;
    double best[2] = { 0.0, 0.0 };
    for (int which = 0; which < 2; ++which)
        for (int rep = 0; rep < 6; ++rep) {
            const int iters = which == 0 ? 1 << 14 : 1 << 12;
            CU(cudaEventRecord(e0, stream()));
            if (which == 0) k_dfma_peak<<<blocks, 256, 0, stream()>>>(out, iters, 0.999999, 1e-9);
            else k_dmma_peak<<<blocks, 256, 0, stream()>>>(out, iters, 0.999999, 1e-9);
            ++g_launches;
            CU(cudaEventRecord(e1, stream()));
            CU(cudaEventSynchronize(e1));
            float ms = 0.f;
            CU(cudaEventElapsedTime(&ms, e0, e1));
            const double fl = which == 0 ? 2.0 * 16.0 * (double)iters * 256.0 * (double)blocks
                                         : 8.0 * 512.0 * (double)iters * 8.0 * (double)blocks;
            if (rep > 0) best[which] = fmax(best[which], fl / (ms * 1e-3) / 1e12);
        }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    dfree(out);
    if (dfma_tflops) *dfma_tflops = best[0];
    if (dmma_tflops) *dmma_tflops = best[1];
    return 0;
}

int fp64_peak(double *tflops)
{
    double a = 0.0, b = 0.0;
    if (fp64_peaks(&a, &b)) return -1;
    *tflops = fmax(a, b);
    return 0;
}

int copy_peak(double *gbs)
{
    const size_t n = (size_t)1 << 30;
    void *a = dmalloc(n), *b = dmalloc(n);
    if (!a || !b) { dfree(a); dfree(b); return -1; }
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
    double best = 0.0;
    for (int rep = 0; rep < 6; ++rep) {
        CU(cudaEventRecord(e0, stream()));
        CU(cudaMemcpyAsync(b, a, n, cudaMemcpyDeviceToDevice, stream()));
        CU(cudaEventRecord(e1, stream()));
        CU(cudaEventSynchronize(e1));
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, e0, e1));
        if (rep > 0) best = fmax(best, 2.0 * (double)n / (ms * 1e-3) / 1e9);
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    dfree(a); dfree(b);
    *gbs = best;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// cross-rank migration: NCCL send/recv over NVLink, resolved at run time from the process's libnccl
// ------------------------------------------------------------------------------------------------
typedef struct { char internal[128]; } nccl_uid;
typedef void *nccl_comm;
struct NcclApi {
    void *lib = nullptr;
    int (*GetUniqueId)(nccl_uid *) = nullptr;
    int (*CommInitRank)(nccl_comm *, int, nccl_uid, int) = nullptr;
    int (*CommDestroy)(nccl_comm) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    int (*Send)(const void *, size_t, int, int, nccl_comm, cudaStream_t) = nullptr;
    int (*Recv)(void *, size_t, int, int, nccl_comm, cudaStream_t) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, nccl_comm, cudaStream_t) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, nccl_comm, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
};
static NcclApi g_nccl;

static int nccl_load()
{
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_nccl.lib) return 0;
    const char *names[] = { "libnccl.so.2", "libnccl.so" };
    for (const char *n : names) { g_nccl.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if (g_nccl.lib) break; }
    if (!g_nccl.lib) { g_be_err = std::string("cannot load libnccl: ") + dlerror(); return -1; }
#define SYM(field, sym) do { *(void **)(&g_nccl.field) = dlsym(g_nccl.lib, sym); if (!g_nccl.field) { g_be_err = std::string("libnccl misses ") + sym; g_nccl.lib = nullptr; return -1; } } while (0)
    SYM(GetUniqueId, "ncclGetUniqueId"); SYM(CommInitRank, "ncclCommInitRank"); SYM(CommDestroy, "ncclCommDestroy");
    SYM(GroupStart, "ncclGroupStart"); SYM(GroupEnd, "ncclGroupEnd"); SYM(Send, "ncclSend"); SYM(Recv, "ncclRecv");
    SYM(AllGather, "ncclAllGather"); SYM(AllReduce, "ncclAllReduce");
    SYM(GetErrorString, "ncclGetErrorString");
#undef SYM
    return 0;
}
#define NC(call) do { int r_ = (call); if (r_ != 0) { g_be_err = std::string(#call) + ": " + g_nccl.GetErrorString(r_); return -1; } } while (0)

int comm_unique_id(uint8_t id[128])
{
    if (nccl_load()) return -1;
    nccl_uid u;
    NC(g_nccl.GetUniqueId(&u));
    memcpy(id, u.internal, 128);
    return 0;
}
// One communicator per (device, rank, n_ranks) is kept for the life of the process: every handle
// of a job that is sharded the same way reuses it (creating one costs about a second), and the
// unique id of later calls is ignored -- all ranks take the same branch, so this stays collective.
struct CommSlot { int rank = -1, n = 0; nccl_comm c = nullptr; };
static CommSlot g_comm[64];

int comm_init(const uint8_t id[128], int rank, int n_ranks, void **comm)
{
    if (nccl_load()) return -1;
    CommSlot &slot = g_comm[g_dev];
    if (slot.c && slot.rank == rank && slot.n == n_ranks) { *comm = slot.c; return 0; }
    nccl_uid u;
    memcpy(u.internal, id, 128);
    nccl_comm c = nullptr;
    NC(g_nccl.CommInitRank(&c, n_ranks, u, rank));
    *comm = c;
    // NCCL opens point-to-point connections lazily: exchange one row with every peer now, so the
    // first migration that crosses ranks does not pay for the connection setup
    if (n_ranks > 1) {
        double *buf = (double *)dmalloc(sizeof(double) * 2 * n_ranks);
        if (!buf) return -1;
        NC(g_nccl.GroupStart());
        for (int r = 0; r < n_ranks; ++r) {
            if (r == rank) continue;
            NC(g_nccl.Send(buf + r, 1, 8 /* ncclFloat64 */, r, c, stream()));
            NC(g_nccl.Recv(buf + n_ranks + r, 1, 8, r, c, stream()));
        }
        NC(g_nccl.GroupEnd());
        CU(cudaStreamSynchronize(stream()));
        dfree(buf);
    }
    if (slot.c && g_nccl.lib) g_nccl.CommDestroy(slot.c);
    slot.rank = rank; slot.n = n_ranks; slot.c = c;
    return 0;
}
int comm_destroy(void *comm)
{
    (void)comm;                                              // owned by the per-device slot above
    return 0;
}
int comm_allgather(void *comm, const void *send, void *recv, size_t bytes_per_rank)
{
    NC(g_nccl.AllGather(send, recv, bytes_per_rank, 0 /* ncclInt8 */, (nccl_comm)comm, stream()));
    return 0;
}
int comm_barrier(void *comm)
{
    static int32_t *buf[64] = { nullptr };
    if (!buf[g_dev]) { CU(cudaMalloc(&buf[g_dev], 2 * sizeof(int32_t))); CU(cudaMemset(buf[g_dev], 0, 2 * sizeof(int32_t))); }
    NC(g_nccl.AllReduce(buf[g_dev], buf[g_dev] + 1, 1, 2 /* ncclInt32 */, 0 /* ncclSum */, (nccl_comm)comm, stream()));
    return 0;
}
__global__ void __launch_bounds__(256) k_pos_from_ids(const int32_t *ids, int n, int32_t *pos)
{
    const int q = blockIdx.x * 256 + threadIdx.x;
    if (q < n) { const int id = ids[q]; if (id >= 0 && id < n) pos[id] = q; }
}
int launch_pos_from_ids(const int32_t *ids, int32_t n, int32_t *pos)
{
    k_pos_from_ids<<<(n + 255) / 256, 256, 0, stream()>>>(ids, n, pos);
    LAUNCHED("k_pos_from_ids");
    return 0;
}
int comm_exchange(void *comm, int rank, int n, const int *src_rank, const int *dst_rank, double *stage_send,
                  double *stage_recv, int row_len)
{
    // position i consumes row r = i-1 (cyclic), produced on src_rank[i], consumed on dst_rank[i]
    NC(g_nccl.GroupStart());
    for (int i = 0; i < n; ++i) {
        if (src_rank[i] == dst_rank[i]) continue;
        const int r = (i + n - 1) % n;
        if (rank == src_rank[i]) NC(g_nccl.Send(stage_send + (size_t)r * row_len, (size_t)row_len, 8 /* ncclFloat64 */, dst_rank[i], (nccl_comm)comm, stream()));
        if (rank == dst_rank[i]) NC(g_nccl.Recv(stage_recv + (size_t)r * row_len, (size_t)row_len, 8 /* ncclFloat64 */, src_rank[i], (nccl_comm)comm, stream()));
    }
    NC(g_nccl.GroupEnd());
    return 0;
}

} // namespace be
} // namespace de

// backend.h -- the device side of libdemcmc_b200 as seen by the host engine: memory, streams and
// one launcher per kernel.  kernels.cu implements it with CUDA for sm_100a.  (tests/emu/ holds a
// host-only test double of the same interface so the engine's host logic can be unit-tested on a
// machine without a GPU; it is never built into or loaded by the product.)
#pragma once
#include <stddef.h>
#include <stdint.h>
#include "de_types.h"

namespace de {
namespace be {

const char *name();                       // "cuda-sm100a" or "emu"
int device_count();
int set_device(int dev);                  // 0 or error
const char *last_error();

void *dmalloc(size_t bytes);              // nullptr on failure (stream-ordered pool)
void *dmalloc_shared(size_t bytes);       // plain device memory that peers write into (the outputs a multi-device handle assembles on one GPU)
void dfree_shared(void *p);
void dfree(void *p);
void *hmalloc_pinned(size_t bytes);
void hfree_pinned(void *p);
int h2d(void *dst, const void *src, size_t bytes);         // on the engine stream, async if src pinned
int d2h(void *dst, const void *src, size_t bytes);         // synchronous
int d2d(void *dst, const void *src, size_t bytes);
int dzero(void *dst, size_t bytes);
int sync();

// lanes: independent kernel chains on separate streams (lane 0 = the engine stream).  set_lane
// selects where the launchers below enqueue; lane_fork makes lanes 1..n-1 wait for everything
// enqueued on lane 0 so far, lane_join makes lane 0 wait for the other lanes.
constexpr int MAX_LANES = 4;          // the persistent chunk kernel interleaves the levels of up to 4 lanes; kernel-chain lanes use 2
void set_lane(int lane);
int lane_fork(int n_lanes);
int lane_join(int n_lanes);

void *event_create();
void event_destroy(void *ev);
int event_record(void *ev);               // on the engine stream
int event_wait(void *ev);                 // host waits

void *tevent_create();                    // timing-capable event
void tevent_destroy(void *ev);
int tevent_elapsed(void *a, void *b, double *ms);
int dfill(void *dst, int byte, size_t bytes);

// CUDA-event stopwatch on the engine stream
int timer_start();
int timer_stop(double *ms);

// ---- kernels ----------------------------------------------------------------------------------
// centres MVN / hierarchical data and packs them for k_xdot (fills center, xT, ssd_xx, ssd_rowmax);
// pack_ssd_doubles = size of the xT buffer the caller must allocate for the model's geometry
size_t pack_ssd_doubles(const ModelDev &m);
// center_host: nullptr = centre on the column means, else the [ssd_k] vector to centre on (host memory)
int launch_pack_ssd(const double *x_in, int in_on_device, const double *center_host, ModelDev *m /* xT allocated */);
// demcmc_eval_pointwise / demcmc_loo: out[i][n] = log p(y_(obs0 + i) | theta_s) for observations [obs0, obs0 + n_obs) of the
// model and the n draws theta[n][d] (device), observation-major (k_ll_obs, k_ll_custom_obs behind ModelDev.custom)
// Declared weak, like the custom-likelihood entry points below: the plain host-only test double does not define these
// two, they resolve to null there, and the engine refuses the model-comparison calls with DEMCMC_EUNSUPPORTED
// (tests/emu/emu_loo.cpp holds host versions that tests/test_loo.py builds into a test double of its own).
int launch_pointwise(const ModelDev &m, const double *theta, int64_t n, int64_t obs0, int64_t n_obs, double *out_obs_major) __attribute__((weak));
// PSIS-LOO and WAIC of each observation from ll[n_obs][n_draws] (device, 2 <= n_draws <= PSIS_MAX_DRAWS): the four outputs
// [n_obs] (device), as include/demcmc_b200.h: demcmc_loo defines them (k_psis)
int launch_psis(const double *ll, int64_t n_draws, int64_t n_obs, double *elpd_loo, double *pareto_k, double *lppd, double *p_waic) __attribute__((weak));
// init_particle: weights of n particles theta[n][d] -> w[n] (also demcmc_eval)
// xdot (MVN / hierarchical, may be nullptr): the cross term of every vector as the likelihood kernel produced it
int launch_eval(const ConfigDev &cfg, const ModelDev &m, const double *theta, int64_t n, double *ll, double *prior,
                double *w, double *scratch_part, double *xdot = nullptr);
// select_base preparation on the sweep-start weights: cw[P] running sums, tot[G]; th[P] is scratch
int launch_base_prep(const ConfigDev &cfg, const double *w, double *th, double *cw, double *tot);
// fills ctxs[s].plan[0..P_local) for the n_sw sweeps of a chunk (contexts with plan == NULL are skipped)
int launch_plan(const ConfigDev &cfg, const SweepCtx *d_ctxs, int n_sw);
// propose -> loglik -> accept for one level of one sweep
int launch_propose(const ConfigDev &cfg, const ModelDev &m, const Level &lv);
// MVN / hierarchical: adds the cross term into ll_acc (fixed point, see de_math.h: xd_scale; launch_propose
// has cleared it and set ll_q); the other models write ll_part
int launch_loglik(const ConfigDev &cfg, const ModelDev &m, const double *theta, const Level &lv, double *ll_part, long long *ll_acc);
int launch_accept(const ConfigDev &cfg, const ModelDev &m, const Level &lv);
// user-written likelihoods (M_CUSTOM): custom_compile builds a DEMCMC_CUSTOM source into an sm_100a cubin with NVRTC and
// keeps it in a per-process cache keyed by the source text (no device needed).  0; -1 = the source does not compile (the
// compiler log is last_error()); -2 = unsupported (no NVRTC, DEMCMC_NPAR above CUSTOM_MAX_PAR, no CUDA backend).
// custom_load loads the source's cubin (compiled first if needed; the same codes, -3 = the CUDA load failed) on the current
// device; launch_loglik
// then runs it for ModelDev.custom = *module.  custom_unload frees a module no launch is still using.
// Declared weak: a backend without a run-time compiler (the host-only test double) does not define them, they resolve to
// null there, and the engine refuses custom models with DEMCMC_EUNSUPPORTED.
int custom_compile(const char *source) __attribute__((weak));
int custom_load(const char *source, void **module, int *has_obs /* the source defines demcmc_obs */) __attribute__((weak));
void custom_unload(void *module) __attribute__((weak));
// simulation-based likelihoods (M_SIMULATED): sim_compile / sim_load are custom_compile / custom_load for a DEMCMC_SIMULATED
// source (its own kernel text k_ll_sim / k_ll_sim_obs; cached apart from a custom source of the same text); the module is
// freed with custom_unload.  launch_loglik and launch_pointwise run it for ModelDev.custom = *module, with the keys of
// include/demcmc_b200.h: DEMCMC_SIMULATED.  launch_eval_sim is launch_eval (ll, prior) with the explicit keys (sweep[n],
// unit[n]) (device) and, when sims is not nullptr, the simulations sims[n][n_sim][n_cols] (device).  Weak, like custom_*.
int sim_compile(const char *source) __attribute__((weak));
int sim_load(const char *source, void **module) __attribute__((weak));
int launch_eval_sim(const ConfigDev &cfg, const ModelDev &m, const double *theta, int64_t n, const uint32_t *sweep, const uint32_t *unit,
                    double *ll, double *prior, double *sims, double *scratch_part) __attribute__((weak));
// small pointwise problems: propose + likelihood + accept of a level in one launch, one warp per
// particle; returns 1 when the model / size does not qualify (launch the three kernels instead)
int launch_level_fused(const ConfigDev &cfg, const ModelDev &m, const Level &lv);
// every level of a chunk of a SMALL pointwise problem (population of at most a few warps) in one single-CTA launch;
// level l = entries [level_off[l], level_off[l + 1]) of d_order.  Returns 1 when the chunk does not qualify.
int launch_chunk_small(const ConfigDev &cfg, const ModelDev &m, const int32_t *d_order, const SweepCtx *d_ctx, const int32_t *level_off, int n_levels);
// all levels of a chunk in ONE persistent, warp-specialised launch (MVN / hierarchical): level l
// holds the entries d_order[level_off[l] .. + level_n[l]); its proposals wait for the accepts of
// level dep[l] (< l, or -1); the scalar warps run their accepts `lag` levels behind their proposals.
// Returns 1 when the chunk does not fit that kernel (launch it level by level instead), -1 on error.
int chunk_persist_lanes(const ConfigDev &cfg, const ModelDev &m);   // lanes that kernel wants for this job; 0 = use the level-by-level path
// n_buf: staging copies of the means (= lanes): level l stages into copy l % n_buf once level l - n_buf has been accepted
int launch_chunk_persist(const ConfigDev &cfg, const ModelDev &m, const int32_t *d_order, const SweepCtx *d_ctx,
                         const int32_t *level_off, const int32_t *level_n, const int32_t *dep, int n_levels, int lag, long long *ll_acc, int n_buf = 2);
// migration (migration.jl:11-116): picks, then gather to / scatter from a staging buffer laid out
// [position][d+3] = {theta..., weight, id, accept flag}
int launch_mig_pick(const ConfigDev &cfg, const MigArgs &a, const double *w, int32_t *picks /*[MAX_MIG]*/);
int launch_mig_gather(const ConfigDev &cfg, const MigArgs &a, const int32_t *picks, const double *theta, const double *w,
                      const int32_t *id, const uint8_t *acc, double *stage);
// pos: id -> position map of the row being edited (resample), or nullptr.  mbox != nullptr: rows whose source is
// another rank (a.src_rank[i] != rank) are taken from slot `slot` of this rank's mailbox once their flag shows `tag`
int launch_mig_scatter(const ConfigDev &cfg, const MigArgs &a, const int32_t *picks, const double *stage, double *theta,
                       double *w, int32_t *id, uint8_t *acc, int32_t *pos, const Mbox *mbox = nullptr, int rank = 0,
                       int slot = 0, unsigned long long tag = 0);
// P2P migration: rows of `stage` produced on this rank and consumed on another are stored into the consumer's mailbox
// (peer-mapped) and published with `tag`
int launch_mig_push(const ConfigDev &cfg, const MigArgs &a, const double *stage, const PeerTable &peers, const Mbox &geom,
                    int rank, int slot, unsigned long long tag);
int mbox_create(int depth, int max_rows, int row_len, Mbox *out);     // plain cudaMalloc (IPC-capable), flags zeroed
void mbox_destroy(Mbox *m);
int mbox_export(const Mbox &m, uint8_t handle[128]);                  // two cudaIpcMemHandle_t
int mbox_open(const uint8_t handle[128], Mbox *peer);                 // maps a peer process's mailbox here
void mbox_close(Mbox *peer);
int enable_peer_access(int dev, int peer_dev);                        // 0, or -1 when the pair has no P2P path
// history rows [n_rows][P][d] by slot -> reference layout [P][d][n_rows] by id (utilities.jl:34)
int launch_history_by_id(const double *rows_theta, const double *rows_w, const uint8_t *rows_acc, const int32_t *rows_id,
                         int64_t n_rows_dev, int64_t row0, int64_t n_rows_out, int32_t P, int32_t d, int32_t id_base,
                         double *samples, double *lp, uint8_t *accept, int32_t P_ids = 0);
// (P = slots per stored row of THIS shard; P_ids = particle ids the outputs cover, id - id_base in [0, P_ids), 0 => P.
// The shards of a multi-device handle pass the whole job's id range and write into one output through peer access.)
// bundle_samples layout (main.jl:222-250): chains[P][d+2][n_rows] for history rows [row0, row0+n_rows);
// final_id[P] = id at each final position, pos_scratch[P] device scratch
int launch_chains(const double *rows_theta, const double *rows_w, const uint8_t *rows_acc, const int32_t *rows_id,
                  const int32_t *final_id, int32_t *pos_scratch, int64_t row0, int64_t n_rows, int32_t P, int32_t d, int32_t id_base, double *out,
                  int32_t P_ids = 0, int32_t pos_base = 0, int phase = 3);
// (phase 1: pos_scratch[id] = pos_base + final position of id; phase 2: the rows; 3: both.  A multi-device handle runs
// phase 1 on every shard, then phase 2 on every shard, all on one pos_scratch[P_ids] and one output.)
// pooled per-parameter mean and sum of squared deviations of n vectors x[n][d] (fixed reduction order)
int launch_moments(const double *x, int64_t n, int32_t d, double *mean, double *m2 /* device [d] each */);
// Convergence diagnostics on the device (SURVEY 8f-1: no download of the draws): every particle id is a chain over
// history rows [row0, row0 + n_rows); each chain is split in two halves of nh = n_rows / 2 draws (the middle one is
// dropped when n_rows is odd).  launch_diag_pos fills pos[r][id] = pos_base + slot for the ids a shard holds at row r
// (ids migrate between shards: every shard writes into the same map); launch_diag_aggregates then gathers every chain
// through that map from the shards' rows.  Output agg[d][3 + n_lag] (device), per flattened parameter k, summed over
// the 2 P_ids split chains in a fixed order: [0] sum of the chain variances (ddof 1), [1] sum of the chain means,
// [2] sum of their squares, [3 + t] sum of the biased autocovariances at lag t < n_lag.  The host turns them into
// split-R-hat and ESS (engine.cpp: diag_finish).
int launch_diag_pos(const int32_t *rows_id, int64_t row0, int64_t n_rows, int32_t P_local, int32_t id_base, int32_t P_ids, int32_t pos_base, int32_t *pos);
int launch_diag_aggregates(const DiagShards &sh, const int32_t *pos, int64_t row0, int64_t n_rows, int32_t P_ids, int32_t d, int32_t lag0, int32_t n_lag, double *agg);   // lags [lag0, lag0 + n_lag)
// Power posteriors.  Declared weak, like launch_pointwise: a backend without them (the plain host-only test double) leaves
// them null, and the engine refuses demcmc_set_temperatures with DEMCMC_EUNSUPPORTED (tests/emu/emu_power_posterior.cpp
// holds host versions that tests/test_power_posterior.py builds into a test double of its own).
// k_power_posterior: the stored untempered log-likelihoods ll_rows[row][P_local] of rows [row0, row0 + n_rows), cut into
// slices of PP_ROWS rows of one local group; part[G_local][n_slices][PP_OUT] (device) gets each slice's
// [count, mean, m2, max, sum e, sum e^2], e = exp(delta.v[g] (ll - slice max)) (de_types.h: PP_OUT).
int launch_power_posterior(const double *ll_rows, int64_t row0, int64_t n_rows, int32_t P_local, int32_t Np, int32_t G_local,
                           const PPDelta &delta, double *part) __attribute__((weak));
// k_temper_weights: the initial weights of a tempered handle, w[p] = prior[p] + tempered_ll(group of p, ll[p]), or -Inf
// where prior[p] is -Inf (out of bounds: launch_eval's prior output), for the n = P_local particles by local position
int launch_temper_weights(const ConfigDev &cfg, const double *prior, const double *ll, int64_t n, double *w) __attribute__((weak));
int diag_max_half();   // longest split chain (stored rows / 2) one call can hold, and
int diag_max_lags();   // the most lags one call computes
// particle algebra known-answer ops (single warp each)
int launch_op_project(const double *p1, const double *p2, int d, double *out);
int launch_op_snooker(const double *pt, const double *pz, const double *pm, const double *pn, double g, const double *b,
                      int d, double *out, double *log_adj);
int launch_op_de(const double *pt, const double *pm, const double *pn, const double *pb, double g1, double g2,
                 const double *b, int d, double *out);
int launch_op_reset(const double *prop, const double *pt, const uint8_t *mask, int d, double *out);
int launch_op_accept(const double *wp, const double *wc, const double *adj, const double *u, int n, uint8_t *out);
int launch_op_select(const double *w, int n, double u, int32_t *base_idx, int32_t *mig_idx);
// roofline probes
int fp64_peak(double *tflops);                             // the larger of the two below
int fp64_peaks(double *dfma_tflops, double *dmma_tflops);   // DFMA loop, DMMA m8n8k4 loop
int copy_peak(double *gbs);

void timeline_dump();                     // debug: writes the %globaltimer stamps of the levels launched so far (DEMCMC_TIMELINE)
int64_t launch_count();                   // kernels launched so far (for demcmc_counters)

// ---- cross-rank migration (NCCL over NVLink) ---------------------------------------------------
int comm_unique_id(uint8_t id[128]);
int comm_init(const uint8_t id[128], int rank, int n_ranks, void **comm);
int comm_destroy(void *comm);
// every rank contributes bytes_per_rank bytes; recv holds the contributions in rank order (resample
// on a sharded job: the replicated copy of a history row)
int comm_allgather(void *comm, const void *send, void *recv, size_t bytes_per_rank);
// device-side barrier on the engine stream: every rank's earlier work has completed before any rank's later work starts
int comm_barrier(void *comm);
// pos[ids[q]] = q for q < n (the id -> position map of a gathered history row)
int launch_pos_from_ids(const int32_t *ids, int32_t n, int32_t *pos);
// grouped send/recv of stage rows: for each position i, src_rank[i] sends row send_pos[i] to dst_rank[i]
int comm_exchange(void *comm, int rank, int n, const int *src_rank, const int *dst_rank, double *stage_send,
                  double *stage_recv, int row_len);

} // namespace be
} // namespace de

// de_types.h -- POD argument blocks passed by value to the kernels of libdemcmc_b200.
#pragma once
#include <stdint.h>
#include "de_math.h"

namespace de {

constexpr int MAX_ACC = 8;        // accumulators of LNR / LBA held in registers
constexpr int SSD_TP = 32;        // particles per CTA tile of the MVN / hierarchical likelihood kernel (4 octets)
constexpr int SSD_OCT = 8;        // particles per DMMA column tile: the granularity of a level's padding
constexpr int SSD_TN = 64;        // observations per tile
constexpr int SSD_NJ = 13;        // max DMMA k-steps (4 dimensions each) per dimension split, held in registers
constexpr int SSD_KS = 4 * SSD_NJ; // max dimensions per dimension split
constexpr int PW_TP = 8;          // particles per tile of the pointwise kernels
constexpr int PW_THREADS = 256;

enum ModelKind { M_GAUSSIAN = 0, M_MVNORMAL = 1, M_BINOMIAL = 2, M_LNR = 3, M_LBA = 4, M_HIER = 5, M_RASTRIGIN = 6, M_MVN_FULL = 7,
                 M_CUSTOM = 8 /* user-written per-observation density compiled at run time (kernels.cu: k_ll_custom) */,
                 M_SIMULATED = 9 /* kernel density of user-written simulations compiled at run time (kernels.cu: k_ll_sim) */ };
constexpr int CUSTOM_MAX_PAR = 256;   // d and DEMCMC_NPAR of a custom model (the per-particle values staged in shared memory)
constexpr int PSIS_MAX_DRAWS = 16384; // draws of one demcmc_loo call: k_psis holds an observation's values in 128 KB of shared memory
constexpr int SIM_MAX_DRAWS = 16384;  // simulations per proposal: k_ll_sim sorts them in 144 KB of shared memory
constexpr int SIM_MAX_LABELS = 8;     // labels of n_cols = 2 data (= MAX_ACC)
constexpr uint32_t SIM_SWEEP_EVAL = 0xFFFFFFFFu;   // the sweep of the simulation keys outside a run
constexpr int PSIS_MAX_TAIL = 512;    // >= the tail length ceil(3 sqrt(PSIS_MAX_DRAWS)) = 384, a power of two (bitonic sort)
// the likelihoods that are a sum of squared deviations from per-dimension means (the streamed DMMA kernels k_xdot / k_chunk_persist)
DE_HD bool is_ssd(int kind) { return kind == M_MVNORMAL || kind == M_HIER || kind == M_MVN_FULL; }
enum { UPDATE_MH = 0, UPDATE_MAXIMIZE = 1, UPDATE_MINIMIZE = 2 };
enum { FITNESS_POSTERIOR = 0, FITNESS_FUN = 1 };

// The registered likelihood a handle is bound to (GPULoglike), device-resident.
struct ModelDev {
    int32_t kind, d;
    int64_t n_obs;
    int32_t n_dim, n_per;
    const double *x;          // pointwise kernels: x[n_obs] / rt[n_obs]
    const int32_t *choice;    // LNR/LBA winners (1-based)
    const double *xT;         // MVN/hier kernel: CENTRED data x' = x - center[k], zero padded, packed as DMMA
                              // A fragments (ssd_pack_index below); the host test double keeps xT[ssd_k][ssd_ld]
    const double *center;     // [ssd_k] column means removed from the data
    const double *linv;       // M_MVN_FULL: inverse of the Cholesky factor of the covariance, lower triangular [n_dim][n_dim]: the
                              // kernel streams the WHITENED data y = Linv (x - raw_center) against the whitened means
                              // Linv (mu - raw_center)
    const double *raw_center; // M_MVN_FULL: [n_dim] centre subtracted in data space, before whitening (the column means, or
                              // demcmc_model.center): Linv x and Linv mu are both of size |Linv| |offset| and their difference
                              // would cancel
    double logdet;            // M_MVN_FULL: log det of the covariance
    double ssd_xx;            // sum of the squared centred data
    double ssd_rowmax;        // 2 max_i |x'_i|: bounds every chain of k_xdot (the cross terms of two observation rows)
    int64_t ssd_n, ssd_ld;    // observations per dimension and padded leading dimension
    int32_t ssd_k;            // dimensions (MVN: n_dim; hierarchical: subjects)
    int32_t ssd_nj;           // DMMA k-steps per dimension split = ceil(ksplit_len / 4)
    int32_t ssd_half;         // ksplit_len % 4 == 2: the last k-step is a HALF step -- its two dimensions of BOTH row
                              // tiles of a pair share one A fragment (columns 0-1: first row tile, 2-3: second), the B
                              // fragment repeats the two means (at load time), and the step costs one DMMA instead of two (d = 50:
                              // 25 DMMAs per row pair and octet instead of 26)
    int32_t ssd_qbits;        // fixed-point bits below the per-particle bound (de_math.h: xd_magic)
    int32_t center_given;     // the data were centred on a caller-supplied vector (demcmc_model.center), not on their column
                              // means: the cross term is then not analytically zero (parity tests of k_xdot / k_chunk_persist)
    int32_t debug_corrupt;    // DEMCMC_TEST_CORRUPT (mutation tests: the parity tests of the cross term must FAIL with it):
                              // 1 = B fragments staged with particle and dimension swapped inside a fragment,
                              // 2 = the half k-step of the second row tile packed over the first, 3 = last k-step not staged
    int32_t has_sigma;
    double sigma_acc[MAX_ACC];
    double lba_floor;
    double binom_N, binom_k;
    const Prior *prior;       // [d]
    int32_t prior_has_ref;    // some prior reads another parameter (NORMAL_REF): priors need the whole proposal
    // partition of the likelihood sum: slice s covers observations [s*split_len, ...) x dimension
    // split; fixed by the model alone so the summation order never depends on the GPU count or on
    // how many slices one CTA happens to process
    int32_t n_osplit, n_ksplit, split_len, ksplit_len;
    uint32_t ksplit_magic;    // ceil(2^32 / ksplit_len): k / ksplit_len = umulhi(k, magic) for every dimension index k < 2^32 / ksplit_len
    int32_t n_cols;           // M_CUSTOM: values per observation, x[n_obs][n_cols]
    void *custom;             // M_CUSTOM / M_SIMULATED: the module loaded on this device (be::custom_load / sim_load), host-side handle
    int32_t n_sim;            // M_SIMULATED: simulations per proposal
    int32_t n_lab;            // M_SIMULATED: labels K (n_cols = 2: the largest label of the data; n_cols = 1: 1)
    double sim_floor;         // M_SIMULATED: density floor
    uint64_t sim_seed;        // M_SIMULATED: the handle's seed, the Philox key of the simulations (launch_pointwise has no ConfigDev)
};

// Packed layout of the centred data for k_xdot: element (observation i, dimension k) lives in the
// DMMA m8n8k4 A fragment of (dimension split ks, row pair rp, observation tile, k-step j): lane =
// (i%8)*4 + k%4 holds the two row tiles of the pair side by side, so one LDS.128 feeds two DMMAs
// and a (ks, rp) stream over observation tiles is contiguous (one bulk copy per stage).
DE_HD int64_t ssd_pack_index(int64_t i, int k, int ksplit_len, int nj, int64_t n_tiles, int half)
{
    const int64_t tile = i / SSD_TN;
    const int r = (int)(i % SSD_TN) / 8, row = (int)(i % 8);
    const int ks = k / ksplit_len, kl = k % ksplit_len;
    const int j = kl / 4;
    const int64_t frag = (((int64_t)(ks * 4 + (r >> 1)) * n_tiles + tile) * nj + j) * 32;
    if (half && j == nj - 1) return (frag + row * 4 + (kl % 4) + 2 * (r & 1)) * 2;   // one fragment for both row tiles
    return (frag + row * 4 + (kl % 4)) * 2 + (r & 1);
}

struct ConfigDev {
    int32_t Np, d, G_local, group_begin, proposal, burnin, n_blocks;
    int32_t resample;         // de.sample = resample: donors are (row, id) cells of the history
    int32_t P_hist;           // particle ids per history row the donors are drawn from: all P of the job (a sharded
                              // job keeps a replicated copy of every row, gathered over the ranks after each iteration)
    int32_t update, fitness;  // UPDATE_* / FITNESS_*: mh_update! + compute_posterior!, or the optimize path
    double eps, sigma, kappa, theta_snooker;
    const double *lo, *hi;    // [d]
    const uint8_t *blocks;    // [n_blocks][d]
    uint64_t seed;
    const double *temp;       // [n_groups] power-posterior temperature of each global group (demcmc_set_temperatures), or
                              // NULL: untempered
};

// The state-independent draws of one particle update (kind, donor slots, gammas, the select_base and accept uniforms):
// functions of (seed, sweep, unit) alone, so a whole chunk's worth is drawn by ONE launch before the chunk's levels run
// (k_plan) and the per-level kernels start from a 64-byte record instead of a ~600-instruction Philox chain per warp.
struct alignas(16) PlanRec { int32_t kind, i0, i1, i2, hr0, hr1, hr2, pad; double g1, g2, u_base, u_acc; };

// One sweep (one pass of mutate_or_crossover! over every local group).  State is kept in ROWS:
// the sweep reads row `cur` (immutable while the sweep runs) and writes row `next`; a donor with
// a smaller slot than the target is read from `next`, reproducing the reference's sequential,
// in-place sweep (crossover.jl:12-17, utilities.jl:201-210) level by level.
struct SweepCtx {
    uint32_t sweep;           // iter0*B + block, the Philox sweep coordinate
    int32_t block;            // block index or -1
    int32_t in_burnin;        // de.iter <= de.burnin (crossover.jl:164)
    int32_t replay;           // draws come from the tape
    int32_t exact_base;       // replay: trust idx[.][0] with sequential semantics
    const double *cur_theta; const double *cur_w; const int32_t *cur_id;
    double *next_theta; double *next_w; int32_t *next_id; uint8_t *next_acc;
    const uint8_t *mutate;    // [G_local] this sweep's rand() <= beta (main.jl:200)
    PlanRec *plan;            // [P_local] this sweep's pre-drawn plans (native mode), or NULL: drawn in place
    // select_base on the sweep-start weights (native mode, burn-in, random_gamma): running sums of
    // the sampling weights per group and their totals (crossover.jl:282-289)
    const double *base_cw;    // [P_local]
    const double *base_tot;   // [G_local]
    // tape slices of this sweep, local shard (replay only)
    const uint8_t *t_kind; const int32_t *t_idx; const double *t_g1, *t_g2, *t_uacc, *t_noise; const uint8_t *t_keep;
    const int32_t *t_idx_row; // resample: history row of each donor (t_idx then holds the particle id)
    // resample (crossover.jl:113-124): the history by position, its id -> position map per row, and
    // the number of rows stored before this iteration (de.iter - 1)
    const double *hist_theta; const int32_t *hist_pos; int64_t donor_rows;
    int32_t *next_pos;        // id -> position map of the row being written, or NULL
    // proposal scratch
    double *prop_theta;       // [P_local][d]
    double *prop_prior;       // [P_local]
    double *prop_adj;         // [P_local]
    double *prop_msq;         // [P_local] sum_k m'_k^2 of the proposal (MVN / hierarchical), written with the proposal
    uint8_t *prop_inb;        // [P_local]
    double *ll_part;          // [P_local][n_split] partial sums of the pointwise kernels
    // MVN / hierarchical: the cross term arrives as an order-independent fixed-point sum,
    // total = ll_acc[p] * ll_q[p] (ll_q NaN: the means are not finite)
    long long *ll_acc;        // [P_local]
    double *ll_q;             // [P_local]
    // trace rows of this sweep or NULL
    double *tr_theta, *tr_w, *tr_adj; uint8_t *tr_acc;
    double *tr_xdot;          // MVN / hierarchical: the cross term the likelihood kernel produced for the proposal
    // tempered handle (ConfigDev.temp): the untempered log-likelihood of each particle, kept with theta; else NULL
    const double *cur_ll; double *next_ll;
};

// One launch: the (sweep slot, local position) updates of one dependency level.  Entry encoding:
// (slot << 24) | position; ctxs[slot] is the sweep the update belongs to (nullptr for plain lists
// of positions, e.g. demcmc_eval).
struct Level { const int32_t *order; int32_t n; const SweepCtx *ctxs; };
constexpr int LV_SLOT_SHIFT = 24;
constexpr uint32_t LV_POS_MASK = (1u << LV_SLOT_SHIFT) - 1;

constexpr int MAX_MIG = 128;      // groups in one migration cycle (kernel-parameter block)
constexpr int MAX_RANKS = 16;     // GPUs of one box a job may shard over
struct MigArgs {
    int32_t n;                      // migrating groups
    int32_t groups[MAX_MIG];        // ordered subset (global group ids)
    double u_pick[MAX_MIG];         // uniform of select_particle per position
    int8_t src_rank[MAX_MIG];       // rank that holds the particle position i receives (picked at position i-1, cyclic)
    int8_t dst_rank[MAX_MIG];       // rank that holds the group at position i
};
// The migration mailbox of one rank, as mapped into this process / device: rows[depth][max_rows][row_len] and one
// 64-bit flag per row.  A sender stores the row with ordinary stores over NVLink (peer-mapped memory), fences at system
// scope and publishes the event's tag in the flag; the receiver's scatter kernel acquires the flag.  No host call and no
// collective sits between a rank's chunks, and only the ranks of the cycle ever wait for each other.
struct Mbox { double *rows; unsigned long long *flags; int32_t depth, max_rows, row_len; };
// history rows of every shard of a job (one entry for a single-device handle): global position q lives at slot q % P_local
// of shard q / P_local
struct DiagShards { const double *theta[MAX_RANKS]; int32_t n, P_local; };
struct PeerTable { double *rows[MAX_RANKS]; unsigned long long *flags[MAX_RANKS]; };
// k_power_posterior: the stored log-likelihoods of one group over PP_ROWS consecutive rows are one slice; its six
// partials are [count, mean, m2 = sum (ll - mean)^2, max, sum e, sum e^2], e = exp(delta (ll - max)).  The slices depend
// on the group and the row range alone, so the partials are the same on any number of devices.
constexpr int PP_ROWS = 256;
constexpr int PP_OUT = 6;
struct PPDelta { double v[MAX_MIG]; };   // delta = t_(k+1) - t_k of the rung k of each local group (0 on the last rung)

// the weight's likelihood term of a particle of global group g: t_g loglike, or loglike itself when untempered.  At t = 0
// the term is 0 whatever the likelihood (the prior alone, as L^0 = 1 reads even where L = 0).
DE_HD double tempered_ll(const ConfigDev &cfg, int g, double ll)
{
    if (!cfg.temp) return ll;
    const double t = cfg.temp[g];
    return t == 0.0 ? 0.0 : mul(t, ll);
}

} // namespace de

/*
 * demcmc_b200.h -- C ABI of libdemcmc_b200.so, the B200 (sm_100a) implementation of the
 * population step of itsdfish/DifferentialEvolutionMCMC.jl.
 *
 * The reference has no FFI (pure Julia).  Each entry point below names the reference interface
 * it replaces (file:line under the reference root); INTEGRATION.md shows the Julia `ccall`
 * binding a maintainer would add, and julia/GPULoglike.jl holds it.
 *
 * Conventions: extern "C"; plain pointers and sizes; every function returns 0 on success or a
 * negative DEMCMC_E* code and never throws; demcmc_last_error() returns a thread-local message.
 * The caller owns every host buffer; the library copies in/out during the call and keeps no host
 * pointer.  Device memory belongs to the handle.  A handle is not thread-safe.  There is no CPU
 * fallback: without a CUDA device demcmc_create fails with DEMCMC_ENODEVICE.
 *
 * Layout: P = n_groups*Np particles, position p = g*Np + j (group-major, the order of
 * sample_init, src/main.jl:263-271); d = flattened parameter count in `names` order, column-major
 * inside array parameters (get_names, src/utilities.jl:131-149).  All indices are 0-based.
 */
#ifndef DEMCMC_B200_H
#define DEMCMC_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DEMCMC_ABI_VERSION 8

enum { DEMCMC_OK = 0, DEMCMC_EINVAL = -1, DEMCMC_ENODEVICE = -2, DEMCMC_ECUDA = -3, DEMCMC_ENOMEM = -4,
       DEMCMC_ESTATE = -5, DEMCMC_EUNSUPPORTED = -6, DEMCMC_ECOMM = -7 };

/* GPULoglike kinds: the registered hand-written likelihood kernels (replace the user closures
 * `loglike(data, theta...)`, e.g. Examples/Gaussian_Example.jl:26-28) */
enum { DEMCMC_GAUSSIAN = 0, DEMCMC_MVNORMAL = 1, DEMCMC_BINOMIAL = 2, DEMCMC_LNR = 3, DEMCMC_LBA = 4,
       DEMCMC_HIER_NORMAL = 5,
       DEMCMC_RASTRIGIN = 6 /* the objective of test/optimization_tests.jl:15-23 (optimize path; no data) */,
       DEMCMC_MVNORMAL_FULL = 7 /* sum(logpdf(MvNormal(mu, sigma^2 * Sigma), data)) with a KNOWN full covariance Sigma
                                   (demcmc_model.cov); parameters mu[n_dim], sigma: d = n_dim + 1 (SURVEY 8f-4).  The data are
                                   whitened once through the Cholesky factor (y = L^-1 x), every proposal's mean is whitened
                                   when it is staged (nu = L^-1 mu), and the isotropic kernels stream y against nu */,
       DEMCMC_CUSTOM = 8        /* a likelihood the caller writes in CUDA C++ (demcmc_model.source), compiled at run time for
                                   sm_100a; see the source contract below */,
       DEMCMC_SIMULATED = 9     /* a likelihood estimated from a simulator the caller writes in CUDA C++ (demcmc_model.source):
                                   a Gaussian kernel density of demcmc_model.n_sim simulations per proposal; see below */ };
/* DEMCMC_CUSTOM source contract.  demcmc_model.source is CUDA C++ text (no #include) that defines
 *   demcmc_obs       required (unless n_obs == 0): __device__ double, arguments (const double *par, const double *x): the
 *                    log density of ONE observation; x = that observation's n_cols values (row i of demcmc_model.x)
 *   demcmc_particle  optional: __device__ double, argument (const double *theta): a term added once per particle (constant
 *                    terms, or the whole objective when n_obs == 0)
 *   DEMCMC_NPAR      optional, with demcmc_prepare: __device__ void, arguments (const double *theta, double *par): a
 *                    per-particle precompute hoisted out of the observation loop (e.g. log(sigma)) that fills
 *                    par[DEMCMC_NPAR]; without it par = theta
 * and the log-likelihood of theta[d] is demcmc_obs of (par, x_i) summed over the observations i, plus demcmc_particle of
 * theta.  theta is the flattened parameter vector in `names` order; d and DEMCMC_NPAR are at most DEMCMC_CUSTOM_MAX_PAR.
 * The observations are summed in a fixed order (per thread, then warp, then block, then split), so a value is the same from run to run and on any
 * number of GPUs.  The CUDA math library (exp, log, lgamma, erfc, normcdf, ...) is available; DEMCMC_INF and
 * DEMCMC_NAN are defined.  A custom model takes the level-by-level path only: the fused and persistent kernels are
 * specialised to the registered kinds. */
#define DEMCMC_CUSTOM_MAX_PAR 256
/* DEMCMC_SIMULATED source contract: a probability density approximation (PDA) of a model that can only be simulated
 * (Turner & Sederberg 2014; Holmes 2015; the reference's Binomial_ABC.jl, KDE_Example.jl, Predator_Prey_Example.jl).
 * demcmc_model.source is CUDA C++ text (no #include) that defines
 *   demcmc_simulate  required: __device__ void, arguments (const double *par, demcmc_rng *rng, double *y): ONE synthetic
 *                    observation y[n_cols] drawn under par, its random numbers taken from rng only
 *   DEMCMC_NPAR      optional, with demcmc_prepare, exactly as for DEMCMC_CUSTOM
 * and the text is given demcmc_rng and two generators:
 *   demcmc_uniform   double, argument (demcmc_rng *): uniform on the open interval (0, 1): 53 random bits b, u = b 2^-53
 *                    (b = 0, of probability 2^-53, gives 2^-54)
 *   demcmc_normal    double, argument (demcmc_rng *): standard normal (Box-Muller on two uniforms; the second value of a
 *                    pair is kept for the next call)
 * The data are x[n_obs][n_cols], n_obs >= 1: n_cols = 1, one continuous value per observation; n_cols = 2, (label, value)
 * with the label an integer-valued double in 1..K, K = the largest label of the data <= DEMCMC_SIM_MAX_LABELS (the
 * (choice, RT) form of the sequential-sampling models).  The data are checked on the host (labels integers in range, values
 * finite), so data_on_device is refused.  d and DEMCMC_NPAR are at most DEMCMC_CUSTOM_MAX_PAR.
 *
 * The estimator, for a proposal theta with key (sweep, unit):
 *   1. simulations y_j = demcmc_simulate of (par, rng_j), j < M = demcmc_model.n_sim (16 <= M <= DEMCMC_SIM_MAX_DRAWS).  rng_j
 *      is the Philox4x32-10 stream with key = the handle's seed and counter (c, unit, sweep, 8 + 16 j), c = 0, 1, ... counting
 *      the Philox calls of the stream (two uniforms each): a function of (seed, sweep, unit, j) alone -- not of the level,
 *      the launch geometry, the path or the device count -- and disjoint from the sampler's own streams (their last
 *      counter word is 1..7).  In a run the key is (the sweep, the particle's global position group_begin * Np + j), the
 *      unit of the proposal noise; the initial weights of demcmc_set_state use (DEMCMC_SIM_SWEEP_EVAL, global position),
 *      demcmc_eval, demcmc_eval_pointwise and demcmc_loo use (DEMCMC_SIM_SWEEP_EVAL, index of the vector);
 *   2. groups: G_c = { j : label of y_j is exactly c and the value of y_j is finite }, c = 1..K (n_cols = 1: one group, the
 *      finite values).  Simulations outside every group still count in M, so the density is DEFECTIVE: label c's density
 *      integrates to m_c / M (m_c = |G_c|);
 *   3. bandwidth: a group with m_c >= 2 gets Silverman's rule, the default of KernelDensity.jl:
 *      h_c = 0.9 min(s_c, IQR_c / 1.34) m_c^(-1/5), s_c the sample sd (ddof 1), IQR_c from linearly interpolated quantiles
 *      (numpy's and Julia's default), s_c alone when IQR_c = 0.  A group with m_c < 2, or with h_c zero or not finite, has
 *      no density;
 *   4. density of an observation (c, t): f = sum_{j in G_c} phi((t - v_j) / h_c) / (M h_c), phi the standard normal density
 *      and v_j the value of y_j; ll_i = log(max(f, sim_floor)), or log(sim_floor) when G_c has no density;
 *   5. the log-likelihood is sum_i ll_i.
 * This is the EXACT Gaussian kernel sum over all m_c simulations, not KernelDensity.jl's binned FFT approximation.  Every
 * sum is formed in a fixed order (the group values sorted, per lane, then the warp's xor tree, then the observations in a
 * fixed order), so a value is the same bits from run to run, on any number of devices and whichever kernel computes it.
 * Pseudo-marginal semantics: only proposals are simulated.  The current particle keeps the estimate it was accepted with,
 * as the reference's stored Particle.weight does; it is never re-evaluated.  A simulated model takes the level-by-level
 * path only. */
#define DEMCMC_SIM_MAX_DRAWS 16384
#define DEMCMC_SIM_MAX_LABELS 8
#define DEMCMC_SIM_SWEEP_EVAL 0xFFFFFFFFu   /* the sweep of every key outside a run (a run never reaches this sweep) */
/* (Examples/Guassian_Example_Vector.jl is the Gaussian model with `loglike(data, theta...)` destructuring its arguments:
 * DEMCMC_GAUSSIAN is its kernel, d = 2 whether the two parameters are named separately or as one 2-vector.) */
/* de.update_particle! (src/utilities.jl:201-226): mh_update!, or the greedy maximize! / minimize! of
 * optimize (src/optimize.jl); de.evaluate_fitness! (src/utilities.jl:92-120): compute_posterior!, or
 * evaluate_fun! = the registered kernel alone, no prior, out of bounds = -/+Inf */
enum { DEMCMC_UPDATE_MH = 0, DEMCMC_UPDATE_MAXIMIZE = 1, DEMCMC_UPDATE_MINIMIZE = 2 };
enum { DEMCMC_FITNESS_POSTERIOR = 0, DEMCMC_FITNESS_FUN = 1 };
/* registered prior specs (replace `prior_loglike(theta...)`, e.g. Examples/Gaussian_Example.jl:11-16) */
enum { DEMCMC_PRIOR_FLAT = 0, DEMCMC_PRIOR_NORMAL = 1, DEMCMC_PRIOR_HALFCAUCHY = 2,
       DEMCMC_PRIOR_UNIFORM = 3, DEMCMC_PRIOR_BETA = 4, DEMCMC_PRIOR_NORMAL_REF = 5 };
/* DE.generate_proposal (src/structs.jl:71, src/crossover.jl:154-226) */
enum { DEMCMC_RANDOM_GAMMA = 0, DEMCMC_FIXED_GAMMA = 1, DEMCMC_VARIABLE_GAMMA = 2 };
/* DE.sample (src/structs.jl:74): where the donor particles come from */
enum { DEMCMC_DONORS_CURRENT = 0, DEMCMC_DONORS_HISTORY = 1 };
/* per-particle update kind on the replay tape */
enum { DEMCMC_KIND_DE = 0, DEMCMC_KIND_SNOOKER = 1, DEMCMC_KIND_MUTATION = 2 };

typedef struct {
    int32_t kind;   /* DEMCMC_PRIOR_* */
    int32_t ref;    /* NORMAL_REF: flattened index of the parameter that is the sd */
    double a, b;    /* NORMAL(mean a, sd b); HALFCAUCHY = truncated(Cauchy(a,b),0,Inf); UNIFORM(a,b);
                       BETA(a,b); NORMAL_REF(mean a, sd theta[ref]) */
} demcmc_prior;

/* Binds a model to a registered kernel: the GPULoglike plugin (replaces DEModel's loglike and
 * prior_loglike closures, src/structs.jl:176-189). */
typedef struct {
    int32_t kind;           /* DEMCMC_GAUSSIAN ... */
    int32_t d;              /* flattened parameter count */
    int64_t n_obs;          /* observations / trials */
    int32_t n_dim;          /* MVNORMAL: data dimension; LNR/LBA: accumulators; HIER: subjects */
    int32_t n_per;          /* HIER: observations per subject */
    const double *x;        /* GAUSSIAN x[n_obs]; MVNORMAL x[n_obs][n_dim] (= Julia n_dim x n_obs
                               column-major); LNR/LBA rt[n_obs]; HIER y[n_dim][n_per];
                               BINOMIAL {N, k} */
    const int32_t *choice;  /* LNR/LBA: 1-based winner per trial, else NULL */
    const double *sigma;    /* LNR: sd per accumulator [n_dim], NULL => 1 */
    double lba_floor;       /* LBA density floor (1e-10 in SequentialSamplingModels), 0 disables */
    const demcmc_prior *prior; /* [d], host memory */
    int32_t data_on_device; /* 1: x / choice are device pointers on the handle's device */
    int32_t n_cols;         /* CUSTOM: values per observation, x[n_obs][n_cols] (= Julia n_cols x n_obs column-major);
                               >= 1 when n_obs > 0.  Unused by the registered kinds */
    const double *cov;      /* MVNORMAL_FULL: covariance [n_dim][n_dim] (host memory), symmetric positive definite */
    const double *center;   /* MVNORMAL / HIER_NORMAL: NULL (the default) = the kernel centres the data on their column
                               means, x' = x - mean: the sum of squares is then  sum x'^2 - 2 B + n sum m'^2  with the
                               streamed cross term B = sum_i sum_k x'_ik m'_k ANALYTICALLY ZERO (sum_i x'_ik = 0) -- the
                               most accurate split, and the reason no likelihood value can show whether the O(N d)
                               stream was computed correctly.  center[n_dim] (host memory) centres on THAT vector
                               instead: B is then n (mean - center).m', not zero, and demcmc_get_trace_xdot /
                               demcmc_eval_xdot expose it, which is how the parity tests pin the DMMA kernels.
                               MVNORMAL_FULL: the centre is in data space, c = the column means or center[n_dim].  The
                               data are centred BEFORE they are whitened, y = L^-1 (x - c), and each mean likewise,
                               m' = L^-1 (mu - c); with NULL the y are then centred on their own column means (about 0)
                               and B is analytically zero, with an explicit centre they are not, and
                               B = sum_i y_i . L^-1 (mu - center). */
    const char *source;     /* CUSTOM / SIMULATED: NUL-terminated CUDA C++ source (host memory), see DEMCMC_CUSTOM /
                               DEMCMC_SIMULATED; else NULL */
    int32_t n_sim;          /* SIMULATED: simulations per proposal M, 16 <= M <= DEMCMC_SIM_MAX_DRAWS */
    double sim_floor;       /* SIMULATED: density floor, > 0 (1e-10 by default, as lba_floor) */
} demcmc_model;

/* Mirrors the DE sampler struct field by field (src/structs.jl:57-131). */
typedef struct {
    int32_t abi_version;     /* DEMCMC_ABI_VERSION */
    int32_t n_groups;        /* de.n_groups: groups in the whole job */
    int32_t Np;              /* de.Np (>= 3: samplepair needs two donors besides the target) */
    int32_t d;
    int32_t burnin;          /* de.burnin */
    int32_t n_initial;       /* de.n_initial: prior rows stored before iteration 1 (utilities.jl:35-39) */
    double alpha, beta, eps, sigma, kappa, theta_snooker; /* de.α β ϵ σ κ θsnooker */
    int32_t proposal;        /* DEMCMC_RANDOM_GAMMA ... */
    int32_t n_blocks;        /* 0: blocking_on(de) == false; else blocking on every iteration */
    const uint8_t *blocks;   /* [n_blocks][d] 1 = updated in this block (de.blocks flattened) */
    const double *lo, *hi;   /* [d] de.bounds expanded per element (src/utilities.jl:70-78) */
    uint64_t seed;           /* Philox key of the native draw map */
    int32_t device;          /* CUDA device ordinal */
    int32_t group_begin;     /* first group held by this handle (multi-GPU: groups shard over ranks) */
    int32_t group_count;     /* groups held by this handle; 0 => all */
    int32_t donors;          /* de.sample (src/structs.jl:74): DEMCMC_DONORS_CURRENT = `sample` (donors from the
                                current group, crossover.jl:138-140), DEMCMC_DONORS_HISTORY = `resample`
                                (DE-MCz: donors from de.samples[1:de.iter-1, :, :], crossover.jl:113-124;
                                needs n_initial > 0 and demcmc_set_history; on a sharded job every rank keeps a
                                replicated copy of the history, gathered with ncclAllGather after each
                                iteration and after each migration) */
    int32_t trace;           /* 1: keep per-sweep proposals / proposal weights / log_adj for
                                demcmc_get_trace (parity tests) */
    int32_t store_every;     /* 1 (or 0) = keep every iteration (reference behaviour, utilities.jl:161-180); k > 1 = thinning:
                                only iterations k, 2k, 3k, ... get a row of de.samples (SURVEY 8f-1: configs[4] writes
                                26.5 MB per iteration per GPU).  Every row count of this header (n_rows, row0) then counts
                                STORED rows: n_initial + iterations / k.  sample = resample draws its donors from the
                                stored rows. */
    int32_t update;          /* DEMCMC_UPDATE_*; maximize!/minimize! need theta_snooker == 0 (they take no log_adj:
                                the reference's snooker branch would throw a MethodError, crossover.jl:38) and
                                leave accept / lp untouched (false / 0.0) */
    int32_t fitness;         /* DEMCMC_FITNESS_* */
    int32_t n_devices;       /* 0 / 1: the handle lives on `device`.  N > 1: ONE handle over the N GPUs devices[0..N) of this
                                box, from ONE process: the groups shard over the devices in order (n_groups % N == 0), one
                                host thread of the library drives each device, migration crosses NVLink through peer-mapped
                                mailboxes, and every demcmc_get_* call returns the whole job exactly as a single-device
                                handle would (same chains bit for bit).  This is what replaces the ThreadsX.map over groups
                                of p_update! (src/main.jl:135-148) for a Julia caller: no MPI, no torchrun.  group_begin /
                                group_count must be 0.  With sample = resample every device keeps a replicated copy of the stored rows: after
                                each iteration (and each migration that edits a stored row) the devices store their slice of the
                                row into each other's copy through peer access and meet at a host barrier. */
    const int32_t *devices;  /* [n_devices] CUDA ordinals, all different, with P2P access to each other */
} demcmc_config;

/* Structured replay tape (SURVEY.md Appendix A): the reference's own random draws, recorded
 * after transformation.  Shapes use the WHOLE job's G and P; S = n_iter*max(1,n_blocks);
 * sweep s = iter0*B + block.  Host memory. */
typedef struct {
    const double  *mig_u;       /* [n_iter]     rand() <= alpha       (src/main.jl:85)            */
    const int32_t *mig_n;       /* [n_iter]     0 = no migration      (src/migration.jl:57)       */
    const int32_t *mig_groups;  /* [n_iter][G]  ordered subset        (src/migration.jl:58)       */
    const double  *mig_pick_u;  /* [n_iter][G]  uniform of select_particle (src/migration.jl:93)  */
    const uint8_t *kind;        /* [S][P]       DEMCMC_KIND_*         (main.jl:200, crossover.jl:31) */
    const int32_t *idx;         /* [S][P][3]    DE (base,m,n) / snooker (z,m,n) slots in the group */
    const double  *gamma1;      /* [S][P]       gamma_1 or snooker gamma (crossover.jl:162,249)   */
    const double  *gamma2;      /* [S][P]       gamma_2, 0 after burn-in (crossover.jl:164)       */
    const double  *u_acc;       /* [S][P]       rand() in accept      (src/utilities.jl:57)       */
    const double  *noise;       /* [S][P][d]    b_k or N(0,sigma) draws (crossover.jl:168, mutation.jl:18) */
    const uint8_t *keep;        /* [S][P][d]    recombination restores theta_t,k; NULL if kappa==1 */
    const int32_t *idx_row;     /* [S][P][3]    resample only: 0-based row of de.samples of each donor; idx then
                                                holds the donor's 0-based particle id (the DE base stays a slot) */
} demcmc_tape;

typedef struct {
    int64_t iterations, sweeps, particle_updates, loglike_evals, kernel_launches, levels;
    double device_ms;        /* CUDA-event time of the last run/replay call */
    double loglike_ms;       /* of which: likelihood kernels (0 unless timing was requested) */
    int64_t persistent_chunks; /* chunks (<= 16 overlapped sweeps) that ran as ONE persistent launch */
    int64_t mailbox_events;    /* migrations whose cycle crossed ranks / devices and went through the peer-mapped mailboxes
                                  (0 with the NCCL send/recv exchange, DEMCMC_MIG=nccl) */
    int64_t cross_migrations;  /* migrations whose cycle crossed ranks / devices, whatever the transport */
} demcmc_counters;

typedef struct demcmc_handle demcmc_handle;

const char *demcmc_last_error(void);
int demcmc_abi_version(void);
int demcmc_device_count(void);
const char *demcmc_backend_name(void);   /* "cuda-sm100a" for the product library */

/* DE(; ...) constructor (src/structs.jl:80-131) */
int demcmc_create(const demcmc_config *cfg, demcmc_handle **out);
int demcmc_destroy(demcmc_handle *h);
/* DEModel(; loglike = GPULoglike(...), prior_loglike = ..., data) (src/structs.jl:176-189) */
int demcmc_set_model(demcmc_handle *h, const demcmc_model *model);
/* Compiles a DEMCMC_CUSTOM source for sm_100a with NVRTC (no device needed) and keeps the result in a per-process cache
 * keyed by the source text, so a later demcmc_set_model with the same text does not compile again.  Returns 0, or
 * DEMCMC_EINVAL with the compiler's log (user lines are reported as user.cu(<line>)) copied into log[log_cap] (may be
 * NULL) and into demcmc_last_error(); DEMCMC_EUNSUPPORTED when libnvrtc.so.12 cannot be loaded or DEMCMC_NPAR is above
 * DEMCMC_CUSTOM_MAX_PAR. */
int demcmc_compile_loglike(const char *source, char *log, int64_t log_cap);
/* The same for a DEMCMC_SIMULATED source (cached apart from a DEMCMC_CUSTOM source of the same text). */
int demcmc_compile_simulator(const char *source, char *log, int64_t log_cap);
/* initialize_samples (src/utilities.jl:29-41) when n_initial > 0: rows[n_initial][P][d], row i = the
 * i-th sample_prior() draw of every particle id; they become rows 1..n_initial of de.samples.  A sharded
 * job passes the rows of its own particles, [n_initial][P_local][d] -- unless sample = resample: then (after
 * demcmc_comm_init) every rank passes the rows of ALL ids, rows[n_initial][P_total][d]. */
int demcmc_set_history(demcmc_handle *h, const double *rows);
/* sample_init / init_particle (src/main.jl:263-271, src/utilities.jl:13-22): theta[P_local][d] by
 * position, ids[P_local] (NULL: id = global position).  Evaluates the initial weights on the device.
 * theta may be NULL after demcmc_set_history: the particles then start from samples[1, :, id]
 * (utilities.jl:15). */
int demcmc_set_state(demcmc_handle *h, const double *theta, const int32_t *ids);
/* the `for iter = 1:n_iter ... stepfun(model, de, groups)` loop of _sample (src/main.jl:33-38),
 * i.e. n_iter x step!/pstep! (src/main.jl:84-107), entirely on the device */
int demcmc_run(demcmc_handle *h, int64_t n_iter);
/* same loop, consuming the reference's recorded draws instead of Philox */
int demcmc_replay(demcmc_handle *h, const demcmc_tape *tape, int64_t n_iter);

/* de.samples (src/utilities.jl:29-41,161-180): out[n_rows][d][P_local] in Julia order (row
 * fastest, then parameter, then particle id - group_begin*Np); n_rows = iterations run so far +
 * n_initial; rows < n_initial are the prior rows of demcmc_set_history */
int demcmc_get_samples(demcmc_handle *h, double *out, int64_t n_rows);
/* Particle.accept / Particle.lp (src/structs.jl:202-208, utilities.jl:207-208): [n_rows][P_local],
 * row fastest, column = particle id - group_begin*Np */
int demcmc_get_accept(demcmc_handle *h, uint8_t *out, int64_t n_rows);
int demcmc_get_lp(demcmc_handle *h, double *out, int64_t n_rows);
/* bundle_samples (src/main.jl:222-250) on the device, for rows [row0, row0+n_rows) of de.samples
 * (n_initial rows included, as the reference indexes them; row0 = burnin when discard_burnin): out[n_rows][d+2][P] in Julia order (= C order [P][d+2][n_rows]), the
 * memory layout of the Array the reference hands to MCMCChains.Chains.  Parameter columns of chain c
 * are the draws of particle id c; the last two columns, "acceptance" and "lp", belong to the
 * particle sitting at final position c -- the reference's own by-position quirk (main.jl:232-241). */
int demcmc_get_chains(demcmc_handle *h, int64_t row0, int64_t n_rows, double *out);
/* Checkpoint / resume (SURVEY 8f-4): a handle created from a saved state (demcmc_get_state ->
 * demcmc_set_state with the ids) continues a chain that has already run `iterations_done` iterations:
 * the Philox counters, de.iter <= burnin (crossover.jl:164) and the migration schedule carry on from
 * there, so run(a) + save + resume + run(b) gives the very chain of run(a + b).  History rows of the new
 * handle start at 0.  Before the first run of the handle; not with sample = resample (its donors are
 * rows of the earlier iterations). */
int demcmc_set_iteration(demcmc_handle *h, int64_t iterations_done);
/* blocking_on(de) (src/structs.jl:75, main.jl:137,162) is a function of the sampler evaluated every
 * iteration; the wrapper evaluates it for the iterations to come and passes the result: on[i] != 0 =>
 * iteration i (0-based, counted from the chain's first iteration: demcmc_set_iteration included) runs
 * block_update! over the handle's blocks, else update! with every parameter at once.  Iterations beyond
 * n are blocked.  Without this call every iteration is blocked (the handle was created with blocks). */
int demcmc_set_blocking_schedule(demcmc_handle *h, const uint8_t *on, int64_t n);
/* ... and the weights (Particle.weight, src/structs.jl:205) the saved particles carried, w[P_local] as
 * demcmc_get_state returned them: demcmc_set_state re-evaluates them, which for the pointwise models sums
 * the observations in another order (same value to ~1e-15 relative, not the same bits). */
int demcmc_set_weights(demcmc_handle *h, const double *w);
/* Streaming summary on the device (SURVEY 8f-1: the history, not the compute, is what stops scaling --
 * configs[4] would hand 423 GB of draws to the host): pooled over history rows [row0, row0+n_rows) and all
 * local particles (rows count from the first history row, the n_initial prior rows included, as in
 * demcmc_get_samples and demcmc_get_diagnostics), per flattened parameter k: mean[k] and m2[k] = sum (x - mean[k])^2, with *count =
 * n_rows * P_local draws, i.e. what MCMCChains' mean / std of the pooled chains reduce to
 * (var = m2 / (count - 1)).  Shards of a multi-GPU job merge (count, mean, m2) with Chan's update. */
int demcmc_get_moments(demcmc_handle *h, int64_t row0, int64_t n_rows, int64_t *count, double *mean, double *m2);
/* Convergence diagnostics computed on the device from the stored rows [row0, row0+n_rows) (no download of the draws):
 * per flattened parameter, split-R-hat and effective sample size with every particle id as one chain, each chain split
 * in two halves (Gelman et al., BDA3 11.4-11.5; Stan's estimators: between / within variances of the split chains,
 * autocorrelations from the chain-averaged autocovariances, Geyer's initial monotone sequence) -- what the reference's
 * tests read off MCMCChains.describe (test/gaussian_tests.jl:42-59), minus the rank normalisation of the newer
 * "bulk" variants (that one needs a global sort of all draws; demcmc_b200.diagnostics computes it on the host).
 * 4 <= n_rows <= 49152 per call (a split chain is held in 192 KB of shared memory; the autocovariances are computed in
 * batches of 4096 lags, and a further batch only while some parameter's Geyer sequence is still positive).  Works on a
 * multi-device handle (the shards' aggregates are merged). */
int demcmc_get_diagnostics(demcmc_handle *h, int64_t row0, int64_t n_rows, double *rhat, double *ess);
/* the same history as the device keeps it, rows [row0, row0+n_rows) of the iterations run, by
 * POSITION: theta[n_rows][P_local][d], w[n_rows][P_local] (= lp), ids[n_rows][P_local] (particle id
 * sitting at each position after that iteration), acc[n_rows][P_local]; any pointer may be NULL.
 * This is what a sharded job gathers on the host (ids migrate across ranks). */
int demcmc_get_history_by_slot(demcmc_handle *h, int64_t row0, int64_t n_rows, double *theta, double *w,
                               int32_t *ids, uint8_t *acc);
/* final `groups` (src/main.jl:36,40): theta[P_local][d], weight[P_local], ids[P_local] by position */
int demcmc_get_state(demcmc_handle *h, double *theta, double *weight, int32_t *ids);
/* per-sweep trace of the LAST run/replay call (needs cfg.trace): prop_theta[S][P_local][d],
 * prop_weight[S][P_local], log_adj[S][P_local], accepted[S][P_local]; any pointer may be NULL */
int demcmc_get_trace(demcmc_handle *h, double *prop_theta, double *prop_weight, double *log_adj, uint8_t *accepted);
/* ... and, MVNORMAL / HIER_NORMAL only, what the streamed likelihood kernel (k_xdot / k_chunk_persist) itself
 * produced for every proposal of that call: xdot[S][P_local] = B = sum_i sum_k (x_ik - center_k)(mean_pk - center_k),
 * the cross term of the expanded sum of squares (Multivariate_Guassian_Example.jl:31-33 has no such intermediate:
 * this is a test hook, see demcmc_model.center) */
int demcmc_get_trace_xdot(demcmc_handle *h, double *xdot);
/* migration picks of the last call: slots[n_iter][G] (-1 where the group did not migrate) */
int demcmc_get_migration(demcmc_handle *h, int32_t *slots);
int demcmc_get_counters(demcmc_handle *h, demcmc_counters *out);
/* measurement mode for bench.py: l2_flush_bytes > 0 overwrites a buffer of that size between
 * chunks of overlapped iterations (evicting L2) and makes counters.device_ms the sum of per-chunk CUDA-event times
 * with the flushes excluded; time_loglik brackets every likelihood launch with CUDA events on the
 * launching stream and reports their sum in counters.loglike_ms */
int demcmc_set_timing(demcmc_handle *h, int64_t l2_flush_bytes, int32_t time_loglik);
/* how many consecutive sweeps (iterations without migration) the device may overlap: the tail
 * dependency levels of one sweep share launches with the head levels of the next (default 16;
 * 1 = a barrier after every sweep).  The result does not depend on it. */
int demcmc_set_max_chunk(demcmc_handle *h, int32_t n_sweeps);
/* how many independent sets of groups run as concurrent kernel chains (groups never read each other
 * between migrations, src/main.jl:161-167): with 2 the likelihood kernel of one set can hide the
 * propose / accept latency of the other.  Default 1: since those two kernels were shortened the second
 * chain only adds launches (profiles/README.md).  The result does not depend on it. */
int demcmc_set_lanes(demcmc_handle *h, int32_t n_lanes);

/* compute_posterior! pieces (src/utilities.jl:92-99) for n arbitrary parameter vectors
 * theta[n][d]: loglike[n], prior[n] (prior is -inf when out of bounds); either may be NULL */
int demcmc_eval(demcmc_handle *h, const double *theta, int64_t n, double *loglike, double *prior);
/* the cross term B (see demcmc_get_trace_xdot) of n arbitrary parameter vectors theta[n][d], through k_xdot */
int demcmc_eval_xdot(demcmc_handle *h, const double *theta, int64_t n, double *xdot);
/* DEMCMC_SIMULATED test hook: loglike[n] of n vectors theta[n][d] under the explicit keys (sweep[i], unit[i]) of
 * DEMCMC_SIMULATED step 1 (the value a run computes for a proposal with that key), and, when sims is not NULL, the
 * simulations sims[n][n_sim][n_cols] in j order */
int demcmc_eval_simulated(demcmc_handle *h, const double *theta, int64_t n, const uint32_t *sweep, const uint32_t *unit,
                          double *loglike, double *sims);
/* SURVEY hard part 7: with the data centred on their column means the cross term is analytically zero, so the
 * MVNORMAL / HIER_NORMAL likelihood follows from O(d) sufficient statistics alone.  on = 1 skips the O(N d) stream
 * (k_xdot / k_chunk_persist are not launched; B is taken as 0).  Off by default: the headline metric counts
 * "loglike evals incl.", i.e. every observation streamed for every particle; bench.py reports this mode
 * separately (value_sufficient_stat).  Refused when the model was given an explicit center. */
int demcmc_set_sufficient_stat(demcmc_handle *h, int32_t on);

/* Model comparison: pointwise log-likelihoods, PSIS-LOO and WAIC on the device.
 *
 * An observation is what demcmc_model.n_obs counts: GAUSSIAN x_i; MVNORMAL / MVNORMAL_FULL row x_i, with the log density
 * logpdf(MvNormal(mu, sigma^2 I or sigma^2 Sigma), x_i); HIER_NORMAL y_sj in the subject-major order of demcmc_model.x
 * (n_obs = n_dim * n_per); LNR / LBA one trial; BINOMIAL the single (N, k) (n_obs = 1); CUSTOM row x_i, its log density
 * the value demcmc_obs returns for it; SIMULATED row x_i, its log density ll_i of DEMCMC_SIMULATED step 4 (draw j simulated
 * under the key (DEMCMC_SIM_SWEEP_EVAL, j), so a row sums to the demcmc_eval value of the draw up to the summation order).
 * Priors are left out, and so is the demcmc_particle term of a CUSTOM model (it belongs to no observation).  A model
 * without observations (RASTRIGIN, CUSTOM with n_obs = 0) is refused with DEMCMC_EINVAL; so is an observation range
 * outside [0, n_obs).  Before demcmc_set_model: DEMCMC_ESTATE.
 *
 * demcmc_loo is PSIS as in Vehtari, Simpson, Gelman, Yao & Gabry (2024), written as ArviZ's psislw / _gpdfit / _gpinv
 * with relative efficiency r_eff = 1.  For each observation i, with ll_s = log p(y_i | theta_s), s < S = n:
 *   1. log ratios r_s = -ll_s, shifted by their maximum: x_s = r_s - max r (so max x = 0);
 *   2. tail length M = ceil(min(S / 5, 3 sqrt(S))); cutoff c = max(the (M+1)-th largest x_s, log(DBL_MIN)); the tail is the
 *      n_t draws with x_s > c (n_t = M unless values tie at the cutoff), in increasing (x_s, s) order;
 *   3. n_t <= 4: no smoothing and k-hat = +Inf;
 *   4. otherwise the Zhang & Stephens (2009) fit to the sorted y_j = exp(x_j) - exp(c), j < n_t: m = 30 + floor(sqrt(n_t))
 *      grid points b_g = (1 - sqrt(m / (g + 1/2))) / (3 y_q) + 1 / y_(n_t - 1), g < m, q = floor(n_t / 4 + 1/2) - 1;
 *      kbar_g = mean_j log1p(-b_g y_j); profile l_g = n_t (log(-b_g / kbar_g) - kbar_g - 1); weight w_g = 1 / sum_h
 *      exp(l_h - l_g); weights below 10 DBL_EPSILON are dropped and the rest normalised to sum 1; b = sum_g w_g b_g;
 *      k = mean_j log1p(-b y_j), sigma = -k / b, and the prior adjustment k-hat = (n_t k + 5) / (n_t + 10);
 *   5. if k-hat is finite, the tail value of rank j becomes log(F^-1((j + 1/2) / n_t) + exp(c)), F^-1 the GPD quantile
 *      sigma (expm1(-k-hat log1p(-p)) / k-hat) (sigma (-log1p(-p)) when |k-hat| < DBL_EPSILON), and then every value
 *      above 0 is set to 0;
 *   6. log weights lw_s = x_s - logsumexp(x);
 *   7. elpd_loo[i] = logsumexp_s(lw_s + ll_s), lppd[i] = logsumexp_s(ll_s) - log S, p_waic[i] = sum_s (ll_s - mean ll)^2 / (S - 1),
 *      pareto_k[i] = k-hat.
 * If any of an observation's S values is not finite, its four outputs are NaN (the call still returns 0).  Every sum is
 * formed in a fixed order, so every output is the same bits from run to run and on any number of devices.  A multi-device
 * handle gives each device a contiguous slice of the observations; a rank of a sharded job holds all the data and
 * computes locally. */
/* log p(y_i | theta_j) for n parameter vectors theta[n][d] and observations [obs0, obs0 + n_obs) of the bound model:
 * out[n][n_obs] (Julia: n_obs x n, data fastest, the [data, draw] order ParetoSmooth.psis_loo takes) */
int demcmc_eval_pointwise(demcmc_handle *h, const double *theta, int64_t n, int64_t obs0, int64_t n_obs, double *out);
/* PSIS-LOO and WAIC per observation over the n draws theta[n][d], all observations of the bound model; each output
 * [n_obs] may be NULL.  2 <= n <= DEMCMC_LOO_MAX_DRAWS (DEMCMC_EINVAL below, DEMCMC_EUNSUPPORTED above: thin the draws) */
int demcmc_loo(demcmc_handle *h, const double *theta, int64_t n, double *elpd_loo, double *pareto_k,
               double *lppd, double *p_waic);
#define DEMCMC_LOO_MAX_DRAWS 16384

/* Model comparison: the marginal likelihood log p(y | M) by power posteriors (Friel & Pettitt 2008; Xie, Lewis, Fan, Kuo &
 * Chen 2011; Annis, Evans, Miller & Palmeri 2019).
 *
 * A tempered handle gives each group g of the job a temperature t_g in [0, 1].  A particle's weight is then
 * prior(theta) + t_g loglike(theta) (the prior alone at t_g = 0), or -Inf out of bounds: this is what the Metropolis accept,
 * select_base, demcmc_get_state and the lp column see.  Each particle also carries loglike(theta) untempered; accept keeps
 * it with theta and every stored row stores it.  A rung is a maximal run of consecutive groups at one temperature.  A
 * tempered handle has no migration, so a particle never leaves its rung.  With every t_g = 1 the chains, lp and accept are
 * bit for bit those of an untempered handle.
 *
 * Refused on a tempered handle: alpha > 0 with more than one group (migration would move particles between temperatures);
 * sample = resample; update maximize! / minimize! and fitness = FUN; demcmc_set_weights (the saved particles' untempered
 * log-likelihoods are unknown); a replay tape with a migration.  A DEMCMC_SIMULATED model takes only t = 1: a power of a
 * noisy likelihood estimate breaks the pseudo-marginal target.
 *
 * demcmc_power_posterior, over the stored rows [row0, row0 + n) of every particle of rung k (temperature t_k, n_k = n times
 * the rung's particles, ll_s the stored untempered log-likelihoods), for k < K rungs:
 *   1. mean_ll[k] and var_ll[k] (ddof 1) of the ll_s;
 *   2. ess_ll[k] and rhat_ll[k]: the split-R-hat and ESS of demcmc_get_diagnostics applied to the ll series, with every
 *      particle id of the rung as one chain;
 *   3. for k < K - 1, delta_k = t_(k+1) - t_k and m_k = max_s ll_s: log_ratio[k] = log((1 / n_k) sum_s e_s) + delta_k m_k with
 *      e_s = exp(delta_k (ll_s - m_k)), the stepping-stone ratio log E_(t_k)[L^delta_k]; log_ratio[K - 1] = NaN.
 * The totals need the rung temperatures to increase strictly in group order, from t_0 = 0 to t_(K-1) = 1:
 *   log_z_ti  = sum_(k < K-1) delta_k (mean_ll[k] + mean_ll[k+1]) / 2                 (the trapezoid rule);
 *   log_z_ti2 = log_z_ti - sum_(k < K-1) delta_k^2 (var_ll[k+1] - var_ll[k]) / 12     (Friel, Hurn & Wyse 2014);
 *   log_z_ss  = sum_(k < K-1) log_ratio[k];
 *   se_ti     = sqrt(sum_k w_k^2 var_ll[k] / ess_ll[k]), w_k the trapezoid weights (delta_(k-1) + delta_k) / 2;
 *   se_ss     = sqrt(sum_(k < K-1) var(e) / (ess_ll[k] mean(e)^2)), the delta method for log of a mean of the e_s, with the
 *               ESS of ll standing in for the ESS of e.
 * The standard errors carry the Monte Carlo error only, not the bias of the temperature ladder.  The rows are cut into
 * slices of one group and 256 rows; each slice's count, mean, sum of squared deviations, max and the two exponential sums
 * are formed on the device (k_power_posterior) in a fixed order, and the host merges them in rung, group and slice order,
 * so every output is the same bits from run to run and on any number of devices. */
typedef struct {
    int32_t n_rungs;
    double log_z_ti, log_z_ti2, log_z_ss, se_ti, se_ss;
} demcmc_evidence;
/* t[n_groups of the whole job], each in [0, 1]: after demcmc_set_model, before demcmc_set_state (the initial weights are
 * tempered; DEMCMC_ESTATE otherwise).  Works on multi-device handles and on the ranks of a sharded job. */
int demcmc_set_temperatures(demcmc_handle *h, const double *t, int32_t n);
/* the stored untempered log-likelihoods of a tempered handle, in the layout of demcmc_get_lp; the prior rows (< n_initial)
 * are NaN */
int demcmc_get_loglike(demcmc_handle *h, double *out, int64_t n_rows);
/* the evidence above over the stored rows [row0, row0 + n_rows); the per-rung arrays [cap] may each be NULL.  DEMCMC_ESTATE
 * without temperatures; DEMCMC_EINVAL when cap < the rungs, the rung temperatures are not 0 < ... < 1 increasing, row0 <
 * n_initial, n_rows < 4, or a parameter has a FLAT prior with an infinite bound (the t = 0 rung would sample an improper
 * prior); DEMCMC_EUNSUPPORTED above 49152 rows (as demcmc_get_diagnostics) and on a rank of a sharded job */
int demcmc_power_posterior(demcmc_handle *h, int64_t row0, int64_t n_rows, int32_t cap, demcmc_evidence *out, double *t,
                           double *mean_ll, double *var_ll, double *ess_ll, double *rhat_ll, double *log_ratio);

/* Particle algebra on the device, for the reference's known-answer tests (test/utility_tests.jl):
 * project (utilities.jl:239-246), reset! (crossover.jl:336-352), random_gamma body
 * (crossover.jl:168; pb NULL => fixed/variable form), snooker_update! (crossover.jl:239-257) with
 * adjust_loglike (crossover.jl:268-273), accept (utilities.jl:55-58) */
int demcmc_op_project(int device, const double *p1, const double *p2, int32_t d, double *out);
int demcmc_op_reset(int device, const double *prop, const double *pt, const uint8_t *mask, int32_t d, double *out);
int demcmc_op_de_proposal(int device, const double *pt, const double *pm, const double *pn, const double *pb,
                          double g1, double g2, const double *b, int32_t d, double *out);
int demcmc_op_snooker(int device, const double *pt, const double *pz, const double *pm, const double *pn,
                      double g, const double *b, int32_t d, double *out, double *log_adj);
int demcmc_op_accept(int device, const double *w_prop, const double *w_cur, const double *log_adj,
                     const double *u, int32_t n, uint8_t *out);
/* select_base (crossover.jl:282-289) and select_particle (migration.jl:89-95) on n weights */
int demcmc_op_select(int device, const double *w, int32_t n, double u, int32_t *base_idx, int32_t *migrate_idx);

/* Multi-GPU: groups shard over ranks; the only exchange is migration (src/migration.jl:109-116),
 * done with NCCL over NVLink when the cycle spans devices.  The host passes the NCCL unique id
 * (128 bytes) obtained on rank 0 to every rank by its own means. */
int demcmc_comm_unique_id(uint8_t id[128]);
int demcmc_comm_init(demcmc_handle *h, const uint8_t id[128], int32_t rank, int32_t n_ranks);

/* fp64 FMA peak of the device in TFLOP/s (DFMA microbenchmark; the roofline denominator that
 * MEASURED_PEAKS.json does not carry) and a copy-bandwidth probe in GB/s */
int demcmc_fp64_peak(int device, double *tflops);
/* both fp64 paths separately: the DFMA (CUDA-core) loop and the DMMA m8n8k4 (tensor) loop; they
 * share one pipe on B200 (scripts/probes/probe_dmma.cu), demcmc_fp64_peak returns the larger */
int demcmc_fp64_peaks(int device, double *dfma_tflops, double *dmma_tflops);
int demcmc_copy_peak(int device, double *gbs);

#ifdef __cplusplus
}
#endif
#endif

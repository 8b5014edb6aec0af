/*
 * stellar_rhmc.h  --  C ABI of libstellar_rhmc.so: the B200-native (sm_100a) RHMC leapfrog hot path of the
 * stellar toy model.
 *
 * The reference (jaekor91/HMC-stellar-toy-model) has no FFI of its own: its seam is the Python method surface of
 * the gym classes.  Each entry point below replaces the reference methods named in its comment (file:line into the
 * reference checkout); hmc_stellar_toy_model_b200/_capi.py is the ctypes binding and INTEGRATION.md shows the
 * stub a reference maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success or a negative srhmc_status; nothing throws or aborts across the ABI;
 *     srhmc_last_error() returns a thread-local, human-readable message for the last failure.
 *   - the caller owns every host pointer; the library copies in/out and owns all device memory inside the context.
 *   - a context is bound to one CUDA device and one stream and is NOT thread-safe (one context per host thread;
 *     ctypes releases the GIL so N contexts drive N GPUs from N threads).
 *   - star state: q and p are float64, flat [f, x, y] per star with f in counts, x along image rows (axis 0);
 *     per field they occupy 3*max_stars slots, of which the first 3*nstars[field] are live.
 *   - images are float64 [rows, cols] C-order on the host whatever the device precision.
 *   - there is no CPU fallback: every entry point needs a CUDA device of compute capability 10.x.
 */
#ifndef STELLAR_RHMC_H
#define STELLAR_RHMC_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SRHMC_ABI_VERSION 3

typedef enum srhmc_status {
    SRHMC_OK = 0,
    SRHMC_ERR_INVALID = -1,   /* bad argument */
    SRHMC_ERR_CUDA = -2,      /* CUDA runtime error (message in srhmc_last_error) */
    SRHMC_ERR_NO_DEVICE = -3, /* no usable sm_100 device */
    SRHMC_ERR_TOO_LARGE = -4, /* field does not fit the resident kernel's shared memory */
    SRHMC_ERR_STATE = -5      /* call order (e.g. run before set_data) */
} srhmc_status;

typedef struct srhmc_ctx srhmc_ctx;

/* Snapshot of the gym attributes the path reads at call time (SURVEY.md 8b "state read at call time").
 * Reference: base_class.__init__/default_exp_setup, sampler_RHMC.py:28-75,169-201. */
typedef struct srhmc_config {
    int32_t abi_version;     /* SRHMC_ABI_VERSION */
    int32_t device;          /* CUDA device ordinal */
    int32_t precision;       /* 64: float64 pixels (parity build); 32: float32 pixels, float64 star state */
    int32_t n_fields;        /* independent fields / chains held by this context */
    int32_t num_rows;        /* gym.num_rows */
    int32_t num_cols;        /* gym.num_cols */
    int32_t max_stars;       /* N_max: star slots per field */
    int32_t patch_radius;    /* 0: full-image PSF (reference semantics); r>0: PSF truncated to (2r+1)^2 pixels */
    int32_t shared_data;     /* 1: one data image shared by all fields (many chains on the same D) */
    int32_t fixed_point_mode;/* 0: reference stop rule (max over the whole field); 1: per-star early exit */
    int32_t use_prior;       /* gym.use_prior */
    int32_t use_Vc;          /* gym.use_Vc */
    double psf_fwhm_pix;     /* gym.PSF_FWHM_pix; sigma = fwhm/2.354 (utils.py:480) */
    double B_count;          /* gym.B_count */
    double f_lim;            /* gym.f_lim */
    double f_low;            /* mag2flux_converter(mB+2): clamp of H_xx (sampler_RHMC.py:267) */
    double g0, g1, g2;       /* utils.factors constants (frozen at 48x48 by the reference) */
    double g_xx, g_ff;       /* metric scale factors */
    double alpha;            /* prior exponent (sampler_RHMC.py:326,409) */
    double V_prior_const;    /* gym.V_prior_const (sampler_RHMC.py:320-321) */
    double Vc_r_pow;         /* repulsion exponent (sampler_RHMC.py:349,417) */
    int32_t enable_hessian;  /* 1: reserve the second shared-memory image the Hessian path needs (srhmc_hessian,
                                SRHMC_LS_HESS); FP64 contexts only */
    int32_t reserved0;
} srhmc_config;

/* samplers.lightsource_gym family: one chain per field with injected draws (the reference's np.random order is
 * p_sample() once, then per iteration p_sample(), randint(steps_min, steps_max), random(); samplers.py:507,520,529,562).
 * Shapes (F fields, S = 3*max_stars, L = niter+1): q0 [F,S]; dt [S] per-coordinate (HMC, HESS, TRIAL) or [1] global
 * (DIAG); normals [F,L,S] (row 0 = the initial p_sample; TRIAL ignores row 0); steps [F,niter]; lnu [F,niter];
 * background [F,R,C] (TRIAL: HMC_find_best_dt's model_data, replaces the constant B) or NULL;
 * outputs (any may be NULL): q_chain [F,L,S], E_chain, dE_chain [F,L], A_chain [F,niter], q_final [F,S],
 * accept_count [F]. */
typedef enum srhmc_ls_variant {
    SRHMC_LS_HMC = 0,   /* lightsource_gym.HMC_random        samplers.py:460-572 */
    SRHMC_LS_DIAG = 1,  /* lightsource_gym.RHMC_random_diag  samplers.py:668-825 */
    SRHMC_LS_HESS = 2,  /* lightsource_gym.RHMC_random       samplers.py:930-1105 */
    SRHMC_LS_TRIAL = 3  /* one acceptance-rate trial of HMC_find_best_dt  samplers.py:327-370, 395-432 */
} srhmc_ls_variant;

typedef struct srhmc_ls_args {
    int32_t variant;
    int32_t niter;
    const double* q0;
    const int32_t* nstars;
    const double* dt;
    int32_t n_dt;
    int32_t zero_xy_momentum;  /* TRIAL: the flux-only tuning pass zeroes p_x, p_y (samplers.py:343-344) */
    double f_lim;              /* gym.f_lim of the run (samplers.py:482-485) */
    double factor1;            /* gym.factor1 (DIAG mass matrix, samplers.py:592-600) */
    const double* normals;
    const int32_t* steps;
    const double* lnu;
    const double* background;
    double* q_chain;
    double* E_chain;
    double* dE_chain;
    uint8_t* A_chain;
    double* q_final;
    double* accept_count;
} srhmc_ls_args;

/* Arguments of one resident chain run.  Replaces the move-0 leg of multi_gym.run_RHMC
 * (sampler_RHMC.py:1009-1083): all (niter+1) x nsteps leapfrog steps, the momentum refresh, the energies and the
 * Metropolis test execute inside ONE kernel launch with no host round trip.
 * Array shapes (F = n_fields, S = 3*max_stars, L = niter+1):
 *   q0 [F,S]; nstars [F] or NULL (= max_stars everywhere);
 *   normals [F,L,S] standard-normal draws replacing np.random.randn (NULL -> device Philox4x32-10, `seed`);
 *   lnu [F,L] log-uniform draws replacing log(np.random.random(1)) (NULL -> device Philox);
 *   g_ff2_schedule [n_g_ff2] / beta_schedule [n_beta] or NULL (sampler_RHMC.py:1011-1016);
 *   outputs (any may be NULL): q_chain, p_chain [F,Ls,S]; E_chain, V_chain, T_chain [F,Ls]; A_chain [F,Ls] uint8
 *   where Ls = ceil(L / chain_stride) rows are kept (row r = iteration r*chain_stride; stride 1 = reference). */
typedef struct srhmc_run_args {
    const double* q0;
    const int32_t* nstars;
    int32_t niter;
    int32_t nsteps;
    double dt;
    double delta;
    int32_t counter_max;
    int32_t f_pos;
    double g_ff2;
    double beta;
    const double* g_ff2_schedule;
    int32_t n_g_ff2;
    const double* beta_schedule;
    int32_t n_beta;
    const double* normals;
    const double* lnu;
    uint64_t seed;
    int32_t chain_stride;
    int32_t reserved;
    double* q_chain;
    double* p_chain;
    double* E_chain;
    double* V_chain;
    double* T_chain;
    uint8_t* A_chain;
    double* q_final;       /* [F,S] state after the last iteration (accepted or restored), may be NULL */
    double* accept_rate;   /* [F] fraction of accepted iterations, may be NULL */
    /* Global identity of the context's fields for the device RNG: field i draws the Philox stream of chain
     * field_id_base + i * field_id_stride (0 / 0 means base 0, stride 1).  A batch sharded over GPUs as
     * ids[rank::world] passes base = rank, stride = world and reproduces the single-GPU run bit for bit. */
    int32_t field_id_base;
    int32_t field_id_stride;
    /* Optional explicit ids [F] overriding base/stride (any shard map).  Note: the one-star kernel packs
     * srhmc_chain_group_size() consecutive fields into a warp and its row windows / log tiers are the union over the
     * warp, so bit-identity with an unsharded run additionally needs shards made of whole groups (sharding.py does that);
     * otherwise results agree to ~1e-15 relative. */
    const int32_t* field_ids;
} srhmc_run_args;

int srhmc_abi_version(void);
const char* srhmc_last_error(void);
int srhmc_device_count(void);
/* Chains the one-star kernel packs into one warp.  Shards of a batch that keep groups of this many consecutive chains
 * together reproduce the unsharded run bit for bit (see srhmc_run_args.field_ids). */
int srhmc_chain_group_size(void);

int srhmc_create(const srhmc_config* cfg, srhmc_ctx** out);
int srhmc_destroy(srhmc_ctx* ctx);

/* Adopt an external CUDA stream (e.g. torch.cuda.current_stream().cuda_stream); 0 restores the context's own. */
int srhmc_set_stream(srhmc_ctx* ctx, void* cuda_stream);
int srhmc_synchronize(srhmc_ctx* ctx);
/* Device time (ms, CUDA events on the launching stream) of the most recent kernel launch of this context. */
int srhmc_last_kernel_ms(srhmc_ctx* ctx, float* ms);
/* Number of kernels this context has launched since creation. */
int64_t srhmc_launch_count(srhmc_ctx* ctx);

/* Pinned host memory helpers for callers that want asynchronous copies. */
void* srhmc_host_alloc(uint64_t bytes);
int srhmc_host_free(void* p);

/* gym.D: n_images = n_fields, or 1 when cfg.shared_data. */
int srhmc_set_data(srhmc_ctx* ctx, const double* D, int64_t n_images);

/* Model image of every field on the device: Lambda = B + sum_s f_s PSF_s.  Replaces base_class.gen_model
 * (sampler_RHMC.py:101-117).  q [F,S] with f in counts; model [F,R,C] (host, written). */
int srhmc_gen_model(srhmc_ctx* ctx, const double* q, const int32_t* nstars, double* model);

/* Mock data on the device: model image of q_true, then one Poisson variate per pixel; the images become the context's
 * data as if passed to srhmc_set_data.  Replaces base_class.gen_mock_data (sampler_RHMC.py:77-99; samplers.py:44-67)
 * with utils.poisson_realization (utils.py:488-496).  The reference draws from NumPy's global stream; here pixel p of
 * field i uses Philox4x32-10 with key `seed` and the 64-bit counter (field_id_base + i) * R * C + p, so a batch sharded
 * over contexts / GPUs gets the same images as an unsharded one (algorithm: NumPy legacy Poisson -- multiplication
 * method below lambda = 10, Hoermann's PTRS above).  D_out [F,R,C] may be NULL (data stay on the device). */
int srhmc_gen_mock_data(srhmc_ctx* ctx, const double* q_true, const int32_t* nstars, uint64_t seed, int64_t field_id_base,
                        double* D_out);

/* One evaluation per field.  Replaces base_class.V (sampler_RHMC.py:294-351), dVdq (:365-425), H with grad
 * (:229-292) and, composed by the caller, dphidq/dtaudq/dtaudp (:448-492); also lightsource_gym.V/dVdq
 * (samplers.py:1108-1150) with use_prior = use_Vc = 0.
 * q [F,S]; outputs (any may be NULL): V [F] (inf outside the support when f_pos / bounds apply),
 * grad [F,S] = dV/dq incl. prior and repulsion, H [F,S], Hgrad [F,S]. */
int srhmc_eval(srhmc_ctx* ctx, const double* q, const int32_t* nstars, int32_t f_pos, double g_ff2, double beta,
               double* V, double* grad, double* H, double* Hgrad);

/* Diagonal metric alone (no image needed).  Replaces base_class.H / H_xx / H_ff (sampler_RHMC.py:229-292).
 * q [n_stars*3] flat [f,x,y] triples (any count, independent of the context's field shape);
 * H, Hgrad [n_stars*3] = [H_ff,H_xx,H_xx] and their d/df (either may be NULL). */
int srhmc_metric(srhmc_ctx* ctx, const double* q, int64_t n_stars, double g_ff2, double* H, double* Hgrad);

/* Kinetic part per field.  Replaces base_class.T (sampler_RHMC.py:353-363), dtaudq (:467-483), dtaudp (:485-492).
 * q, p [F,S]; outputs (any may be NULL): T [F] = (sum p^2/H + sum ln|H|)/2 with H = H(q), dtaudq [F,S], dtaudp [F,S]. */
int srhmc_kinetic(srhmc_ctx* ctx, const double* q, const double* p, const int32_t* nstars, double g_ff2,
                  double* T, double* dtaudq, double* dtaudp);

/* T for an explicit diagonal H_diag, as base_class.T(p, H_diag) takes it (sampler_RHMC.py:353-363): p, H_diag [n]. */
int srhmc_kinetic_diag(srhmc_ctx* ctx, const double* p, const double* H_diag, int64_t n, double* T);

/* nsteps generalised-leapfrog steps in place.  Replaces base_class.RHMC_single_step (sampler_RHMC.py:522-566).
 * fp_counts, if not NULL, receives [F,2]: the two fixed-point iteration counts of the LAST step. */
int srhmc_step(srhmc_ctx* ctx, double* q, double* p, const int32_t* nstars, int32_t nsteps, double dt,
               double delta, int32_t counter_max, double g_ff2, double beta, int32_t* fp_counts);

/* Full chain (see srhmc_run_args).  srhmc_run = upload + launch + download + synchronize.  The three phases are
 * also exported so a caller can keep inputs resident and time the launch alone. */
int srhmc_run(srhmc_ctx* ctx, const srhmc_run_args* args);
int srhmc_run_upload(srhmc_ctx* ctx, const srhmc_run_args* args);
int srhmc_run_launch(srhmc_ctx* ctx, const srhmc_run_args* args);
int srhmc_run_download(srhmc_ctx* ctx, const srhmc_run_args* args);

/* One long trajectory per field recording V-V0, T-T0 and their sum after every step.  Replaces
 * single_gym.run_single_RHMC(solver="implicit") (sampler_RHMC.py:649-783).
 * q0, p0 [F,S]; q_chain, p_chain [F,nsteps+1,S]; E_chain, V_chain, T_chain [F,nsteps+1] (row 0: q0,p0, zeros). */
int srhmc_run_single(srhmc_ctx* ctx, const double* q0, const double* p0, const int32_t* nstars, int32_t nsteps,
                     double dt, double delta, int32_t counter_max, int32_t f_pos, double g_ff2, double beta,
                     double* q_chain, double* p_chain, double* E_chain, double* V_chain, double* T_chain);

/* lightsource_gym chains (see srhmc_ls_args).  Contexts for these calls are created with use_prior = use_Vc = 0. */
int srhmc_ls_run(srhmc_ctx* ctx, const srhmc_ls_args* args);

/* Replaces lightsource_gym.RHMC_efficient_computation (samplers.py:828-927).  q, p [F,S]; f_lim as gym.f_lim;
 * d2_only != 0: only d2 = dVdqq is produced and the flux floor is not checked (the reference's dVdqq_only=True);
 * otherwise d1 = dVdq, d2, d3 = dVdqqq, dqdt, dpdt [F,S] and E [F] (all +inf when a flux is below f_lim).
 * Needs enable_hessian = 1 at context creation. */
int srhmc_hessian(srhmc_ctx* ctx, const double* q, const double* p, const int32_t* nstars, double f_lim, int32_t d2_only,
                  double* d1, double* d2, double* d3, double* dqdt, double* dpdt, double* E);

/* Potential and gradient of the fields' stars on a per-pixel background image replacing the constant B.  Replaces
 * lightsource_gym.V_single / dVdq_single (samplers.py:77-127) with max_stars = 1 (background = model_data).
 * q [F,S]; background [F,R,C]; V [F] = -sum(D ln Lambda - Lambda); grad [F,S]. */
int srhmc_eval_background(srhmc_ctx* ctx, const double* q, const int32_t* nstars, const double* background, double* V,
                          double* grad);

/* Gradient-descent leg of lightsource_gym.find_peaks (samplers.py:196-226): each of the n seeds q_seed [n,3] (f, x, y;
 * updated in place) descends independently on the context's data image (field 0) over a pure-background model with the
 * steps dt_f = f dt_f_coeff, dt_xy = dt_xy_coeff / f, until |dV/V| < 1e-9, nstep steps, or f < f_lim (alive[i] = 0).
 * V_single / dVdq_single (samplers.py:77-127) are evaluated device-side, one warp per seed, one launch for all seeds.
 * steps_taken [n] may be NULL.  The grid seeding and the final merge stay with the caller (samplers.py:160-178, 234-252). */
int srhmc_find_peaks_descend(srhmc_ctx* ctx, double* q_seed, int32_t n, int32_t nstep, double dt_f_coeff, double dt_xy_coeff,
                             double f_lim, uint8_t* alive, int32_t* steps_taken);

/* Split-chain Gelman-Rubin statistic and effective sample size per variable.  Replaces utils.convergence_stats (with
 * utils.variogram), utils.py:86-188, including its definitions of W (mean of the within-chain standard deviations) and
 * of the autocorrelation cut-off.  q_chain [n_chains, n_iter, d] on the host; the chains form n_groups consecutive groups
 * of n_chains / n_groups chains (one call of the reference per group); R, n_eff [n_groups, d]. */
int srhmc_convergence_stats(int32_t device, const double* q_chain, int64_t n_chains, int64_t n_iter, int32_t d, int32_t n_groups,
                            int32_t thin_rate, int32_t warm_up_num, double* R, double* n_eff);
/* The same statistics over the q_chain of the context's last launched run, which is still resident on the device
 * (srhmc_run_upload + srhmc_run_launch with q_chain requested; srhmc_run_download is not needed): a batch of thousands of
 * chains returns 2 * n_groups * 3 * max_stars numbers instead of its chains.  Rows are the stored rows of the run
 * (chain_stride applied).  R, n_eff [n_groups, 3 * max_stars]. */
int srhmc_run_stats(srhmc_ctx* ctx, int32_t n_groups, int32_t thin_rate, int32_t warm_up_num, double* R, double* n_eff);

/* Draws of the device generator, for replaying a Philox run through another implementation:
 * normals [F,L,S], lnu [F,L] exactly as srhmc_run would consume them for `seed`. */
int srhmc_philox_draws(srhmc_ctx* ctx, uint64_t seed, int32_t niter, double* normals, double* lnu);
/* Same with the global field identity of srhmc_run_args. */
int srhmc_philox_draws_ids(srhmc_ctx* ctx, uint64_t seed, int32_t niter, int32_t field_id_base, int32_t field_id_stride,
                           double* normals, double* lnu);

/* Diagnostic (host only, no device needed): into how many iteration chunks the one-star kernel's work scheduler cuts a
 * run of n_iterations (= niter + 1) Metropolis iterations for `groups` warp-sized groups of chains on `resident_warps`
 * warps -- n_parts = 0: a single launch; n_parts > 0: the pipelined srhmc_run of that many launches (returns the total
 * over the parts, 0 if impossible).  Every chunk of ceil(n_iterations / chunks) iterations is non-empty. */
int srhmc_plan_chunks(int64_t groups, int64_t resident_warps, int32_t n_iterations, int32_t n_parts);

/* Diagnostic: evaluate the kernels' own device math on n values (which = 0: exp_neg(x), x <= 0; 1: log_pos(x), x > 0;
 * 2: rcp_fast(x)) so the test-suite can bound its error against libm. */
int srhmc_test_device_math(srhmc_ctx* ctx, int32_t which, const double* x, double* y, int32_t n);

/* ------------------------------------------------------------------------------------------------------------------
 * Large-field engine: one crowded field too big for a single CTA, optionally one row-strip of a field tiled over the
 * GPUs of a node (BASELINE configs[2] scaled up, configs[4]).  Same physics as srhmc_step / srhmc_run with use_Vc = 0
 * and a PSF truncated to (2r+1)^2 pixels; replaces the same reference methods (sampler_RHMC.py:229-566, 1009-1083).
 *
 * A rank owns the global rows [own_lo, own_hi) and holds data rows [row0, row0+nrows) = strip + `nrows_halo` rows on
 * each interior side.  One leapfrog step is the phase sequence
 *     KICK1 -> [max-reduce counters] -> PFIX_QFIX -> [max-reduce counters] -> QFIX_KICK -> PACK -> [all-gather
 *     ghost_send into ghost_recv] -> EVAL | EVAL_V -> KICK2
 * (inside a trajectory "EVAL -> KICK2 -> next step's KICK1" is the single phase EVAL_KICK2_KICK1, and the last step ends
 * with EVAL_V_KICK2: four kernels per leapfrog step on one GPU)
 * and one Metropolis iteration is
 *     MOMENTUM -> ENERGY -> [sum-reduce scalars into global_scalars] -> RECORD_E0 -> nsteps x step -> ENERGY ->
 *     [sum-reduce] -> ACCEPT.
 * Every phase only ENQUEUES kernels on the context's stream; the bracketed collectives are issued by the caller on the
 * same stream (torch.distributed / NCCL on tensors wrapping the buffers of srhmc_big_buffers) and are skipped for
 * world_size = 1.  hmc_stellar_toy_model_b200/bigfield.py is the reference orchestration. */
typedef struct srhmc_big srhmc_big;

typedef struct srhmc_big_config {
    int32_t abi_version;
    int32_t device;
    int32_t rows_global, cols;   /* gym.num_rows, gym.num_cols of the whole field */
    int32_t own_lo, own_hi;      /* owned global rows */
    int32_t row0, nrows;         /* local data rows (strip + halo) */
    int32_t nrows_halo;          /* halo rows per interior side (>= patch_radius; the excess is the drift allowance) */
    int32_t max_stars;           /* capacity for owned stars */
    int32_t max_ghosts;          /* capacity of each boundary list */
    int32_t patch_radius;        /* PSF truncation radius r (1..15); r = 12 is within 3e-13 of the full-image PSF */
    int32_t use_prior;
    int32_t world_size, rank;
    double psf_fwhm_pix, B_count, f_lim, f_low, g0, g1, g2, g_xx, g_ff, alpha, V_prior_const;
} srhmc_big_config;

typedef enum srhmc_big_phase_id {
    SRHMC_BIG_PACK = 0,       /* boundary stars -> ghost_send */
    SRHMC_BIG_EVAL = 1,       /* model image, residual, per-star pixel gradient (a2) */
    SRHMC_BIG_EVAL_V = 2,     /* same + pixel potential of the owned rows -> scalars[0] (a3) */
    SRHMC_BIG_KICK1 = 3,      /* p -= h dphi/dq; p fixed point phase A -> counters[0] (a7 steps 1-2) */
    SRHMC_BIG_PFIX_QFIX = 4,  /* p fixed point phase B; q fixed point phase A -> counters[1] (a7 steps 2-3) */
    SRHMC_BIG_QFIX_KICK = 5,  /* q fixed point phase B; p -= h dtau/dq (a7 steps 3-4) */
    SRHMC_BIG_KICK2 = 6,      /* p -= h dphi/dq at the new q; reflections (a7 steps 5-6) */
    SRHMC_BIG_MOMENTUM = 7,   /* p = z sqrt(H); remember the iteration's start state (a8) */
    SRHMC_BIG_ENERGY = 8,     /* scalars[1..3] = T, #stars outside the support, prior potential (a3, a5) */
    SRHMC_BIG_RECORD_E0 = 9,  /* E0 from global_scalars; chain row; sample row while recording (srhmc_big_set_recording) */
    SRHMC_BIG_ACCEPT = 10,    /* Metropolis test on global_scalars; restore on rejection; chain row (a8) */
    SRHMC_BIG_RESET_ITER = 11, /* zero the device-side iteration counter used when step.iteration < 0 */
    /* fused forms (same arithmetic in the same order, fewer launches): */
    SRHMC_BIG_EVAL_KICK2 = 12,       /* EVAL then KICK2 */
    SRHMC_BIG_EVAL_V_KICK2 = 13,     /* EVAL_V then KICK2 */
    SRHMC_BIG_EVAL_KICK2_KICK1 = 14, /* EVAL, KICK2 and the KICK1 of the following leapfrog step (same q, same gradient) */
    /* per-star stop rule (srhmc_big_step.fixed_point_mode = 1): steps 1-4 of a7 couple no stars, so they are one kernel */
    SRHMC_BIG_PS_ADVANCE = 15,       /* KICK1, both fixed points to each star's own convergence, p -= h dtau/dq, binning */
    SRHMC_BIG_EVAL_PS_ADVANCE = 16   /* EVAL, KICK2 and the PS_ADVANCE of the following leapfrog step */
} srhmc_big_phase_id;

typedef struct srhmc_big_step {
    double dt, delta, g_ff2;
    int32_t counter_max, f_pos;
    int32_t iteration;       /* Metropolis iteration index (RNG counter, chain row); < 0: use the device-side counter,
                                which ACCEPT advances -- lets one captured CUDA graph of an iteration be replayed */
    int32_t fixed_point_mode;/* 0: reference stop rule (sampler_RHMC.py:531-545: both implicit loops run until the slowest
                                star of the WHOLE field has converged; tiled over GPUs that is two max all-reduces per
                                leapfrog step); 1: per-star early exit, as srhmc_config.fixed_point_mode = 1 (results differ
                                from the reference by less than `delta` per step; no iteration count crosses the GPUs) */
    uint64_t seed;
} srhmc_big_step;

/* Device pointers of the buffers the caller's collectives operate on (sizes in elements). */
typedef struct srhmc_big_buffers_t {
    void* ghost_send;  int64_t ghost_send_doubles;   /* [2][1 + 3*max_ghosts]: count, then f,x,y triples */
    void* ghost_recv;  int64_t ghost_recv_doubles;   /* [world][2][1 + 3*max_ghosts] (all-gather of ghost_send) */
    void* scalars;                                   /* double[n_scalars]: this rank's partial sums */
    void* global_scalars;                            /* double[n_scalars]: the all-reduced sums */
    int64_t n_scalars;
    void* counters;    int64_t n_counters;           /* int32[n_counters]: fixed-point iteration counts (max-reduce) */
} srhmc_big_buffers_t;

const char* srhmc_big_last_error(void);
int srhmc_big_create(const srhmc_big_config* cfg, srhmc_big** out);
int srhmc_big_destroy(srhmc_big* b);
int srhmc_big_set_stream(srhmc_big* b, void* cuda_stream);    /* NULL = the CUDA default stream; a new context runs on
                                                                  its own non-blocking stream until this is called */
int srhmc_big_adopt_stream(srhmc_big* b, void* cuda_stream);  /* no synchronisation: usable during graph capture */
int srhmc_big_synchronize(srhmc_big* b);
int64_t srhmc_big_launch_count(srhmc_big* b);
int srhmc_big_set_data(srhmc_big* b, const double* D_local /* [nrows, cols] */);
/* 32: the FP32 build -- gradient-only evaluations (every leapfrog step but the last of a trajectory) read a float copy of the
 * data window and render / reduce in float; star state and every evaluation that returns the potential stay FP64.  Needs the
 * tile path (srhmc_big_create chooses it for fields of at least 2 tiles per SM).  64 (default): everything FP64. */
int srhmc_big_set_precision(srhmc_big* b, int32_t precision);
/* Device-side gen_mock_data for the local data window (see srhmc_gen_mock_data): q_true [n,3] (f in counts, x, y) is
 * the WHOLE field's truth list, identical on every rank; the Philox counter is the global pixel index, so halo rows agree
 * between ranks.  D_local_out [nrows, cols] may be NULL. */
int srhmc_big_mock_data(srhmc_big* b, const double* q_true, int32_t n, uint64_t seed, double* D_local_out);
int srhmc_big_set_stars(srhmc_big* b, const double* q /* [n,3] */, const int64_t* global_ids /* [n] */, int32_t n);
int srhmc_big_get_stars(srhmc_big* b, double* q, double* p, double* grad /* each [n,3], may be NULL */);
int srhmc_big_set_momenta(srhmc_big* b, const double* p /* [n,3] */);
int srhmc_big_buffers(srhmc_big* b, srhmc_big_buffers_t* out);
/* Peer exchange: the bracketed collectives above done by the library's own kernels over peer-mapped memory (NVLink P2P
 * between the GPUs of one node) instead of by the caller.  Every rank exports its mailbox (a 64-byte CUDA IPC handle for
 * other processes and/or the raw device pointer for strips hosted by the same process), the caller distributes the
 * handles (any transport: they are plain bytes) and every rank imports all `world_size` of them (ipc_handles: world x 64
 * bytes, or raw_ptrs: world pointers; the own entry is ignored).  From then on the phases that produce the fixed-point
 * counters (KICK1, PFIX_QFIX, EVAL_KICK2_KICK1) all-reduce(max) them themselves, PACK also delivers the boundary lists
 * into the neighbours' ghost_recv, and RECORD_E0 / ACCEPT sum the scalars over the ranks (rank order, identical on every
 * rank): the caller issues no collective, and a captured CUDA graph of an iteration can be replayed on every rank.  A peer
 * that never arrives raises error flag 4 after ~10 s instead of hanging the device. */
int srhmc_big_comm_export(srhmc_big* b, void* ipc_handle_64 /* may be NULL */, void** raw_ptr /* may be NULL */);
int srhmc_big_comm_import(srhmc_big* b, const void* ipc_handles, void* const* raw_ptrs);
/* Parity mode: normals [n_iters, n, 3] for the owned stars and/or lnu [n_iters]; NULL -> device Philox (seed). */
int srhmc_big_set_draws(srhmc_big* b, const double* normals, const double* lnu, int32_t n_iters);
int srhmc_big_alloc_chains(srhmc_big* b, int32_t n_iters);
int srhmc_big_read_chains(srhmc_big* b, int32_t n_iters, double* E, double* V, double* T, uint8_t* A, double* n_accepted,
                          int32_t* error_flag /* 1: an owned star left the local data window; 2: ghost list overflow;
                                                    3: tile list overflow; 4: peer exchange timed out */);
int srhmc_big_read_scalars(srhmc_big* b, double* scalars);
int srhmc_big_phase(srhmc_big* b, int32_t phase, const srhmc_big_step* step);
/* Sample recording (the q_chain / p_chain of multi_gym.run_RHMC): from the next RECORD_E0 on, the phase also stores the owned
 * stars' q (before the trajectory) and/or p (just drawn by MOMENTUM) of iteration l as row l / stride when stride divides l:
 * ceil(n_iters / stride) rows of [n][3] doubles on the device, stars in ascending global-id order (slot order, independent of
 * the storage order).  The iteration index is step.iteration, or the device counter when it is < 0, so eager runs and replays
 * of a captured iteration record alike.  One extra kernel per RECORD_E0 while recording; nothing changes while it is off.
 * want_q = want_p = 0 turns recording off and frees the rows.  Call it after srhmc_big_set_stars and outside graph capture: it
 * may move the buffers. */
int srhmc_big_set_recording(srhmc_big* b, int32_t n_iters, int32_t stride, int32_t want_q, int32_t want_p);
/* Rows [row0, row0 + nrows) of the recorded samples, each [n][3] in slot order (q or p may be NULL): a long chain can be
 * fetched in pieces. */
int srhmc_big_read_samples(srhmc_big* b, int32_t row0, int32_t nrows, double* q, double* p);
/* utils.convergence_stats over k (2..16) chains of the same field: k contexts on one device that own the same global ids and
 * recorded q with the same row count and stride.  thin_rate / warm_up_num apply to the recorded rows.  R, n_eff [3 n] in slot
 * order.  One thread per variable over the resident rows (variable-parallel: few chains, many variables). */
int srhmc_big_convergence_stats(srhmc_big* const* chains, int32_t k, int32_t thin_rate, int32_t warm_up_num, double* R,
                                double* n_eff);

/* Roofline denominator measured on the device itself: a register-resident FMA chain (8 independent chains per
 * thread, all SMs filled) in the given precision (64 or 32).  Returns TFLOP/s (2 flop per FMA) and the launch time. */
int srhmc_measure_fma_peak(int32_t device, int32_t precision, double* tflops, float* ms);

#ifdef __cplusplus
}
#endif
#endif /* STELLAR_RHMC_H */

/*
 * bjx.h -- C ABI of the B200-native HMC/NUTS hot path (libbjx.so).
 *
 * Drop-in boundary for BlackJAX's `blackjax.hmc` / `blackjax.nuts` / `window_adaptation`
 * path (reference: blackjax-devs/blackjax @ 63912a4).  The reference has no FFI of its own
 * (it is pure Python on JAX), so every entry point below cites the reference *function* it
 * replaces; `INTEGRATION.md` shows the ctypes binding a maintainer would add.
 *
 * Conventions
 *  - All array pointers are DEVICE pointers owned by the caller unless marked "host".
 *  - State arrays are row-major float32 [n_chains, dim] (chain-major, dimension contiguous);
 *    per-chain scalars are [n_chains]; PRNG keys are uint32 [n_chains, 2] (raw threefry keys,
 *    i.e. jax.random.key_data layout).
 *  - Every call is asynchronous and ordered on the handle's stream (bjx_nuts_step included: the tree doubling is
 *    driven from host C++ as launches whose row counts stay on the device); the only calls that wait for the
 *    device are bjx_synchronize, bjx_destroy, bjx_nuts_last_stats and -- once per tree doubling -- bjx_nuts_step on the
 *    tensor-core dense path (dense metric / dense target with dim > 128: the products are sized from the row count).
 *  - Dense metrics and dense Gaussian targets are built for dim <= 1024: beyond, bjx_create / bjx_set_metric return
 *    BJX_E_UNSUPPORTED (the tensor-core products would miss their 1e-5 per-product accuracy).
 *  - Return value: 0 ok; <0 invalid argument / unsupported configuration (BJX_E_*);
 *    >0 a cudaError_t.  bjx_last_error(handle) returns the text.  No exceptions or
 *    callbacks cross this ABI.  A handle is not thread-safe; distinct handles are independent.
 *  - There is NO CPU fallback: every entry point fails with a CUDA error if no device exists.
 */
#ifndef BJX_H_
#define BJX_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BJX_VERSION 100

/* error codes (negative) */
#define BJX_OK 0
#define BJX_E_INVALID (-1)     /* bad argument / shape */
#define BJX_E_UNSUPPORTED (-2) /* configuration not built (e.g. dim % 4 != 0 with dim > 128) */
#define BJX_E_STATE (-3)       /* call order (e.g. metric not set) */

/* log-density targets with a fused analytic value_and_grad (replaces jax.value_and_grad of the
 * user callable: blackjax/mcmc/hmc.py:91, integrators.py:189,204). */
enum bjx_target_kind {
  BJX_TARGET_DIAG_GAUSSIAN = 0,  /* -1/2 sum ((x-mean)/s)^2 + offset   tests/fixtures.py:60-78   */
  BJX_TARGET_FUNNEL = 1,         /* Neal's funnel                       tests/fixtures.py:81-98   */
  BJX_TARGET_DENSE_GAUSSIAN = 2, /* -1/2 x^T P x + offset               tests/mcmc/test_mclmc_lrd.py:86-88 */
  BJX_TARGET_BANANA = 3,         /* -(1-x0)^2 - 1.5 (x1-x0^2)^2, dim=2  tests/mcmc/test_trajectory.py:79-80 */
  BJX_TARGET_HIER_LOGIT = 4,     /* hierarchical logistic regression (BASELINE config 5; builder-defined, see
                                    DESIGN.md): x = [mu, log tau, beta0, beta1, alpha_0..alpha_{G-1}], dim = 4 + G */
  BJX_TARGET_USER = 5            /* user-defined value_and_grad compiled into a plug-in (bjx_plugin_load; dim <= 1024):
                                    the slot of the arbitrary `logdensity_fn` callable of hmc.py:91 / nuts.py:133 */
};

/* inverse-mass-matrix layouts (metrics.py:701-729: 1-D => diagonal, 2-D => dense) */
enum bjx_metric_kind {
  BJX_METRIC_DIAG = 0,          /* imm [dim]                                    */
  BJX_METRIC_DENSE = 1,         /* imm [dim, dim] symmetric positive definite   */
  BJX_METRIC_DIAG_PER_CHAIN = 2, /* imm [n_chains, dim] (vmapped window adaptation) */
  BJX_METRIC_LOW_RANK = 3,       /* bjx_set_metric_low_rank */
  BJX_METRIC_DENSE_PER_CHAIN = 4 /* imm [n_chains, dim, dim], dim <= 64 (vmapped dense window adaptation) */
};

typedef struct {
  int32_t kind;           /* bjx_target_kind */
  int32_t dim;
  const float* inv_var;   /* DIAG_GAUSSIAN: [dim] 1/s^2 (device)           */
  const float* mean;      /* DIAG_GAUSSIAN: [dim] or NULL (device)         */
  const float* precision; /* DENSE_GAUSSIAN: [dim, dim] symmetric (device) */
  float logp_offset;      /* constant added to every log-density           */
  const float* data_x;    /* HIER_LOGIT: covariates [G, 8, 2] (device)     */
  const uint8_t* data_y;  /* HIER_LOGIT: outcomes, bit k of byte g = y_gk  */
  int32_t n_groups;       /* HIER_LOGIT: G (dim = 4 + G)                   */
  int32_t n_user_params;  /* USER: floats in user_params                   */
  const float* user_params; /* USER: parameter block (device) or NULL      */
  void* user_plugin;      /* USER: plug-in from bjx_plugin_load            */
} bjx_target_desc;

typedef struct {
  int32_t device;              /* CUDA ordinal */
  int32_t n_chains;            /* chains held by THIS process/GPU */
  int32_t dim;
  int32_t max_tree_depth;      /* NUTS checkpoint capacity (max_num_doublings upper bound), >= 1 */
  float divergence_threshold;  /* default 1000 (hmc.py:120, trajectory.py:325) */
  void* stream;                /* cudaStream_t to order all work on (NULL = legacy default stream) */
  bjx_target_desc target;
} bjx_config;

/* Optional per-transition outputs (NULL => not written).  Mirrors HMCInfo (hmc.py:52-87) and
 * NUTSInfo (nuts.py:36-74); D-sized fields only on request. */
typedef struct {
  float* acceptance_rate;          /* [C]                                              */
  uint8_t* is_accepted;            /* [C]   HMC only                                   */
  uint8_t* is_divergent;           /* [C]                                              */
  uint8_t* is_turning;             /* [C]   NUTS only                                  */
  float* energy;                   /* [C]   energy of the proposal                     */
  int32_t* num_integration_steps;  /* [C]                                              */
  int32_t* num_trajectory_expansions; /* [C] NUTS only                                 */
  float* momentum;                 /* [C,D] momentum drawn at the start of the transition */
  float* proposal_position;        /* [C,D] HMC: end state (before accept/reject)      */
  float* proposal_momentum;        /* [C,D] HMC: flipped end momentum                  */
  float* left_position;            /* [C,D] NUTS trajectory_leftmost_state.position    */
  float* left_momentum;            /* [C,D]                                            */
  float* right_position;           /* [C,D] NUTS trajectory_rightmost_state.position   */
  float* right_momentum;           /* [C,D]                                            */
} bjx_info;

typedef struct bjx_handle_s* bjx_handle_t;

/* ---- lifecycle ------------------------------------------------------------------------------ */
int bjx_version(void);
int bjx_create(const bjx_config* cfg, bjx_handle_t* out);
int bjx_destroy(bjx_handle_t h);
const char* bjx_last_error(bjx_handle_t h); /* h may be NULL: last global error */
int bjx_set_target(bjx_handle_t h, const bjx_target_desc* target);
/* User-defined targets.  BlackJAX takes any callable and differentiates it (`jax.value_and_grad(logdensity_fn)`,
 * mcmc/hmc.py:91, integrators.py:189); here the plug-in point is the fused value_and_grad device function
 * (`bjx_user::Model<R>::value_and_grad`, contract in include/bjx_user_target.h).  A plug-in is a small shared library built from
 * blackjax_b200/csrc/bjx_plugin.cu + the user's source (nvcc; blackjax_b200/plugin.py does it from Python) holding every
 * transition kernel of the path instantiated around that function.  bjx_plugin_load opens it (host path), checks that it
 * was built against this library's kernel ABI (bjx_plugin_abi) and returns the pointer to put into
 * bjx_target_desc.user_plugin with kind = BJX_TARGET_USER.  Plug-ins stay loaded for the life of the process. */
int bjx_plugin_load(const char* path, void** plugin_out);
int bjx_plugin_abi(void);
/* Palindromic two-stage integrator (integrators.py:62-152): host array of n coefficients, n odd in 3..11.
 * {0.5, 1, 0.5} = velocity_verlet (default, :321-322); mclachlan :335-340, yoshida :351-357, omelyan :363-369. */
int bjx_set_integrator(bjx_handle_t h, const float* coefficients, int32_t n);
/* Key source for bjx_sample_momentum / bjx_hmc_step / bjx_mhmc_step / bjx_nuts_step: shared_step_key = 0 (default):
 * `keys` is uint32 [n_chains, 2], one rng_key per chain.  shared_step_key = 1: `keys` is ONE key uint32 [2] and
 * chain c uses jax.random.split(key, n_global)[chain_offset + c] (= fold_in(key, chain_offset + c)), derived inside the
 * kernel -- the reference's step-major schedule (docs/examples/howto_sample_multiple_chains.md:116-129), independent
 * of how the chains are sharded over GPUs (chain_offset = first global chain of this handle). */
int bjx_set_key_mode(bjx_handle_t h, int32_t shared_step_key, uint32_t chain_offset);
/* Dynamic HMC (blackjax/mcmc/dynamic_hmc.py:62-130): every chain integrates its own number of steps.  steps_dev: int32
 * [n_chains] device array read by the following bjx_hmc_step / bjx_mhmc_step calls (their scalar L is then ignored);
 * NULL restores the scalar.  The caller keeps the array alive until those calls have run.  dim <= 1024 only. */
int bjx_set_integration_steps(bjx_handle_t h, const int32_t* steps_dev);
/* Generalized HMC slice noise (mcmc/ghmc.py:90,172 `noise_fn(key_noise)`, key_noise = split(rng_key)[1]): per-chain values
 * float32 [C] (device) for the following bjx_ghmc_step calls, evaluated by the caller; NULL = the default noise_fn (0). */
int bjx_set_ghmc_noise(bjx_handle_t h, const float* noise_dev);
int bjx_synchronize(bjx_handle_t h);

/* metrics.default_metric / gaussian_euclidean (metrics.py:180-218,221-346): precomputes
 * mass_matrix_sqrt = 1/sqrt(M^-1) (diag) or L^-T with L = chol(M^-1) (dense), metrics.py:701-729.
 * The dense factorisation runs on the host in float64 and synchronises the stream.  Dense: dim <= 1024. */
int bjx_set_metric(bjx_handle_t h, int32_t metric_kind, const float* inverse_mass_matrix);
/* metrics.gaussian_euclidean_low_rank(sigma, U, lam) (metrics.py:349-467): M^-1 = diag(sigma) (I + U (Lambda - I) U^T) diag(sigma),
 * sigma [dim] > 0, U [dim, rank] row-major with orthonormal columns, lam [rank] > 0 (device arrays, copied).  Momentum
 * draw, kinetic energy, velocity and the U-turn test all cost O(dim * rank).  rank <= 16, dim <= 512 (warp kernels: HMC,
 * multinomial HMC, NUTS). */
int bjx_set_metric_low_rank(bjx_handle_t h, const float* sigma, const float* U, const float* lam, int32_t rank);
/* device pointer to mass_matrix_sqrt as precomputed by bjx_set_metric (for tests) */
int bjx_get_mass_matrix_sqrt(bjx_handle_t h, const float** out);

/* ---- building blocks (KAT-able; each maps to one reference function) -------------------------- */
/* hmc.init (hmc.py:90-92): logp, grad = value_and_grad(logdensity)(q) */
int bjx_init_state(bjx_handle_t h, const float* q, float* logp_out, float* grad_out);
/* metric.sample_momentum (metrics.py:260-261 -> util.py:66-91): p = mass_matrix_sqrt (.) normal(key,(D,)) */
int bjx_sample_momentum(bjx_handle_t h, const uint32_t* keys, float* p_out);
/* static_integration (trajectory.py:136-167) of velocity_verlet (integrators.py:62-152,321-322):
 * n_steps leapfrogs in place.  step_size_dev ([C], signed) overrides step_size when non-NULL. */
int bjx_leapfrog(bjx_handle_t h, float* q, float* p, float* logp, float* grad, float step_size,
                 const float* step_size_dev, int32_t n_steps);
/* linear_map(inverse_mass_matrix, p) (blackjax/util.py:23-61; the kinetic-energy gradient of
 * integrators.py:242): v = M^-1 p for every chain.  Dense metric with dim > 128: one tensor-core GEMM. */
int bjx_metric_velocity(bjx_handle_t h, const float* p, float* v_out);
/* hmc_energy (trajectory.py:730-750): -logp + 1/2 p^T M^-1 p */
int bjx_energy(bjx_handle_t h, const float* p, const float* logp, float* energy_out);
/* metrics.is_turning (metrics.py:272-304) on explicit momenta (for the U-turn truth table) */
int bjx_is_turning(bjx_handle_t h, const float* p_left, const float* p_right, const float* p_sum,
                   uint8_t* out);

/* ---- transitions ------------------------------------------------------------------------------ */
/* hmc.build_kernel(...).kernel (hmc.py:279-312).  (q,logp,grad)_in -> (q,logp,grad)_out; out may
 * alias in (in-place).  keys: one rng_key per chain. */
int bjx_hmc_step(bjx_handle_t h, const uint32_t* keys, const float* q_in, const float* logp_in,
                 const float* grad_in, float* q_out, float* logp_out, float* grad_out,
                 float step_size, const float* step_size_dev, int32_t num_integration_steps,
                 const bjx_info* info);
/* Multinomial HMC: hmc.build_kernel(build_proposal=multinomial_hmc_proposal) = blackjax.mhmc (hmc.py:181-248,
 * trajectory.py:170-232, blackjax/__init__.py:145-151).  Same arguments as bjx_hmc_step; is_accepted is always 1,
 * acceptance_rate = exp(sum_log_p_accept) / L, proposal_* = the selected trajectory state. */
int bjx_mhmc_step(bjx_handle_t h, const uint32_t* keys, const float* q_in, const float* logp_in,
                  const float* grad_in, float* q_out, float* logp_out, float* grad_out,
                  float step_size, const float* step_size_dev, int32_t num_integration_steps,
                  const bjx_info* info);
/* Generalized HMC: ghmc.build_kernel().kernel (blackjax/mcmc/ghmc.py:118-189; update_momentum :192-213;
 * nonreversible_slice_sampling blackjax/mcmc/proposal.py:243-264), in place on the persistent state
 * (q [C,D], p [C,D], logp [C], grad [C,D], slice [C]); noise_fn is the reference default (0).
 * step_size_dev / alpha_dev / delta_dev (optional) are indexed by chain / chains_per_group; imm_rows + msqrt_rows
 * (optional, [C / chains_per_group, D]: inverse mass = momentum_inverse_scale^2, ghmc.py:83-84, and 1/sqrt of it)
 * override the handle's diagonal metric row-wise -- MEADS' per-fold parameters (meads_adaptation.py:587-606).
 * Chains in [skip_begin, skip_end) are computed but keep their state (the frozen fold, :639-650). */
int bjx_ghmc_step(bjx_handle_t h, const uint32_t* keys, float* q, float* p, float* logp, float* grad, float* slice,
                  float step_size, const float* step_size_dev, float alpha, const float* alpha_dev, float delta,
                  const float* delta_dev, const float* imm_rows, const float* msqrt_rows, int32_t chains_per_group,
                  int32_t skip_begin, int32_t skip_end, const bjx_info* info);
/* MEADS fold statistics and parameters (blackjax/adaptation/meads_adaptation.py:507-585, maximum_eigenvalue :787-817)
 * from the positions and gradients of all chains, folds = contiguous blocks of C / num_folds chains, t = the
 * adaptation iteration.  state float32 [bjx_meads_state_floats] = step_size[K] | alpha[K] | delta[K] | sigma[K,D] |
 * imm[K,D] | msqrt[K,D], already rolled by one fold (:560-563), i.e. the arrays bjx_ghmc_step takes.
 * num_folds = 1 gives base.compute_parameters (:97-152) of all chains. */
size_t bjx_meads_state_floats(int32_t num_folds, int32_t dim);
size_t bjx_meads_scratch_floats(int32_t n_chains, int32_t dim, int32_t num_folds);
int bjx_meads_update(bjx_handle_t h, const float* q, const float* grad, int32_t num_folds, int32_t t,
                     float step_size_multiplier, float damping_slowdown, float* state, float* scratch);
/* maximum_eigenvalue (meads_adaptation.py:787-817) of one float32 [n, d] device matrix; out: ONE device float */
size_t bjx_maximum_eigenvalue_scratch_floats(int64_t n, int32_t d);
int bjx_maximum_eigenvalue(bjx_handle_t h, const float* x, int64_t n, int32_t d, float* out, float* scratch);
/* jax.random.permutation(key', n) with key' = fold_in(key, fold_index) (fold_index < 0: key itself): the sort-based
 * shuffle of jax/_src/random.py.  perm_out int32 [n]; scratch: bjx_permutation_scratch_bytes(n) bytes. */
size_t bjx_permutation_scratch_bytes(int64_t n);
int bjx_permutation(bjx_handle_t h, const uint32_t* key, int64_t fold_index, int64_t n, int32_t* perm_out, void* scratch);
/* dst[r, :] = src[perm[r], :] for float32 [rows, width] (the shuffle of meads_adaptation.py:675-683); out of place */
int bjx_gather_rows(bjx_handle_t h, const int32_t* perm, const float* src, float* dst, int64_t rows, int32_t width);
/* blackjax.util.run_inference_algorithm (util.py:150-213) for HMC (multinomial = 0) / multinomial HMC (1), run
 * natively: step keys = jax.random.split(rng_key, num_steps) (util.py:203), num_steps in-place transitions enqueued back
 * to back without host synchronisation; chain c of step t uses split(step_key_t, n_global)[chain_offset + c].
 * rng_key: ONE key uint32 [2] (device).  history (optional): float32 [num_steps / thin, C, D], the positions after every
 * thin-th transition; acceptance_history (optional): float32 [num_steps, C]. */
int bjx_hmc_sample(bjx_handle_t h, const uint32_t* rng_key, float* q, float* logp, float* grad, float step_size,
                   const float* step_size_dev, int32_t num_integration_steps, int32_t num_steps, int32_t multinomial,
                   float* history, int32_t thin, float* acceptance_history);
/* nuts.build_kernel(...).kernel (nuts.py:113-145) with iterative_nuts_proposal (nuts.py:223-321).
 * Tree doubling is driven from the host: one launch per doubling over the chains still expanding; each
 * warp integrates its chain's whole sub-tree (up to 2^d leapfrog leaves) inside the launch.
 * Dense metric / dense Gaussian target with 128 < dim <= 1024: the chains of a doubling advance through its leaves in lock
 * step, compacted, on the tensor-core products (three per leaf: half-step velocity, gradient, full-step velocity for the
 * energy and the U-turn tests, metrics.py:263-304); same keys and decisions.
 * momentum_override/key_integrator_override (both or neither, for KATs): skip the key split and
 * the momentum draw and use the given momentum [C,D] and integrator keys [C,2]. */
int bjx_nuts_step(bjx_handle_t h, const uint32_t* keys, const float* q_in, const float* logp_in,
                  const float* grad_in, float* q_out, float* logp_out, float* grad_out,
                  float step_size, const float* step_size_dev, int32_t max_num_doublings,
                  const bjx_info* info, const float* momentum_override,
                  const uint32_t* key_integrator_override);
/* blackjax.util.run_inference_algorithm (util.py:150-213) for NUTS, run natively like bjx_hmc_sample: step keys =
 * split(rng_key, num_steps), transitions in place, no host synchronisation.  With num_steps >= 4 the chains run DECOUPLED:
 * one persistent launch whose warps take whole chains through all transitions (chains never interact and transition t
 * of chain c needs only step key t), bit-identical to num_steps calls of bjx_nuts_step.  history (optional) float32
 * [num_steps / thin, C, D]; acceptance_history (optional) float32 [num_steps, C]; num_integration_steps_history (optional)
 * int32 [num_steps, C]. */
int bjx_nuts_sample(bjx_handle_t h, const uint32_t* rng_key, float* q, float* logp, float* grad, float step_size,
                    const float* step_size_dev, int32_t max_num_doublings, int32_t num_steps, float* history, int32_t thin,
                    float* acceptance_history, int32_t* num_integration_steps_history);
/* doubling launches and the deepest tree of the last bjx_nuts_step (host ints; reading the depth synchronises the stream) */
int bjx_nuts_last_stats(bjx_handle_t h, int64_t* doubling_launches, int64_t* depth_reached);

/* ---- PRNG (jax.random restated; keys raw uint32 pairs) ----------------------------------------- */
/* h may be NULL for the PRNG entry points: current device, and the stream this thread registered with
 * bjx_set_default_stream (a cudaStream_t; the legacy default stream until one is registered) */
int bjx_set_default_stream(void* cuda_stream);
int bjx_prng_split(bjx_handle_t h, const uint32_t* keys, int64_t n_keys, int32_t num, uint32_t* out);
int bjx_prng_fold_in(bjx_handle_t h, const uint32_t* keys, int64_t n_keys, uint32_t data, uint32_t* out);
int bjx_prng_random_bits(bjx_handle_t h, const uint32_t* keys, int64_t n_keys, int64_t per_key, uint32_t* out);
int bjx_prng_uniform(bjx_handle_t h, const uint32_t* keys, int64_t n_keys, int64_t per_key, float* out);
int bjx_prng_normal(bjx_handle_t h, const uint32_t* keys, int64_t n_keys, int64_t per_key, float* out);
/* jax.random.randint(key, shape, minval, maxval) int32 -- dynamic_hmc's default integration_steps_fn
 * (dynamic_hmc.py:66: randint(key, (), 1, 10)) */
int bjx_prng_randint(bjx_handle_t h, const uint32_t* keys, int64_t n_keys, int64_t per_key, int32_t minval, int32_t maxval,
                     int32_t* out);

/* ---- window adaptation (staged_adaptation.py:111-307) -------------------------------------------- */
/* Per-chain dual averaging (optimizers/dual_averaging.py:87-129).  da_state float32 [C,5] =
 * (log_step, log_step_avg, step, avg_error, mu).  step_size_out [C] = exp(log_step). */
int bjx_da_init(bjx_handle_t h, float* da_state, const float* initial_step_size /*[C]*/, float* step_size_out);
int bjx_da_update(bjx_handle_t h, float* da_state, const float* acceptance_rate, float target, float* step_size_out);
/* slow-window end: re-initialise DA at exp(log_step_avg) (staged_adaptation.py:233-249) */
int bjx_da_reset(bjx_handle_t h, float* da_state, float* step_size_out);
int bjx_da_final(bjx_handle_t h, const float* da_state, float* step_size_out);
/* Per-chain diagonal Welford (adaptation/mass_matrix.py:411-442): mean,m2 [C,D]; count is a host int */
int bjx_welford_update(bjx_handle_t h, const float* q, float* mean, float* m2, int32_t new_count);
/* regularised IMM (mass_matrix.py:335-357): imm = n/(n+5) m2/(n-1) + 1e-3*5/(n+5); resets mean,m2 */
int bjx_welford_final(bjx_handle_t h, float* mean, float* m2, int32_t count, float* imm_out);
/* Per-chain dense Welford (mass_matrix.py:411-442 with is_diagonal_matrix=False): mean [C,D], m2 [C,D,D];
 * m2 += outer(x - mean_new, x - mean_old) */
int bjx_welford_dense_update(bjx_handle_t h, const float* q, float* mean, float* m2, int32_t new_count);
/* regularised dense IMM per chain (mass_matrix.py:335-357): imm = n/(n+5) m2/(n-1) + 1e-3*5/(n+5) I; resets mean,m2 */
int bjx_welford_dense_final(bjx_handle_t h, float* mean, float* m2, int32_t count, float* imm_out);
/* Chain-pooled summary block of THIS GPU's chains for the shared-epsilon warm-up
 * (staged_adaptation.py:153-171,906-966; metric_buffers.py:396-420):
 * stats_out float32 [2 + 2*D] = (sum acceptance_rate, n_chains, mean[D], M2[D]).
 * The blocks of all GPUs are exchanged with ONE all-gather and CGL-merged on every rank. */
int bjx_pooled_stats(bjx_handle_t h, const float* q, const float* acceptance_rate, float* stats_out);
/* Dense variant (welford_dense recipe; metric_buffers.py:396-420 `centered.T @ centered`), any dim (float32 SIMT tiles in
 * a fixed order; dim = 512 x 32768 chains: a few ms):
 * stats_out float32 [2 + D + D*D] = (sum acceptance_rate, n_chains, mean[D], M2[D,D]). */
int bjx_pooled_stats_dense(bjx_handle_t h, const float* q, const float* acceptance_rate, float* stats_out);

/* ---- shared (cross-chain, cross-GPU) window adaptation, device resident ------------------------------------------
 * The reference's multi-chain path (staged_adaptation.py:153-171,906-966): ONE dual-averaging update per warm-up step
 * on the mean acceptance rate of ALL chains and, in slow windows, the chain-pooled moment block merged into the window
 * accumulator (metric_buffers.py:334-420); its cross-device collective is lax.psum over "chains" (eca.py:56-62).
 * Here: each GPU reduces its chains in fixed blocks of BJX_STAT_BLOCK_CHAINS chains to (sum accept, n, mean[D], M2[D]),
 * ONE NCCL all-gather exchanges the blocks, and every rank merges them in global chain order and applies the same
 * update on the device -- results do not depend on the GPU count when chains_per_gpu % BJX_STAT_BLOCK_CHAINS == 0. */
#define BJX_STAT_BLOCK_CHAINS 4096
/* NCCL communicator helpers (libnccl.so.2 is bound at run time; single-GPU callers never need it).  A caller that
 * already owns an ncclComm_t (e.g. an XLA / framework communicator) passes it to the calls below as is. */
int bjx_nccl_unique_id(void* id128_out);                      /* ncclGetUniqueId: 128 bytes, on rank 0 */
int bjx_nccl_comm_init_rank(const void* id128, int32_t n_ranks, int32_t rank, int32_t device, void** nccl_comm_out);
int bjx_nccl_comm_destroy(void* nccl_comm);
/* The collective of the path: all-gather `count` floats per rank into gathered[n_ranks * count] on the handle's stream.
 * nccl_comm is an ncclComm_t (NULL: one rank, gathered = block). */
int bjx_allgather_stats(bjx_handle_t h, void* nccl_comm, const float* block, int64_t count, float* gathered);
/* Device state of the shared adaptation: bjx_adapt_shared_state_floats(...) floats (dual averaging, window accumulator,
 * this rank's blocks and the gathered blocks). */
int64_t bjx_adapt_shared_state_floats(int32_t n_chains_local, int32_t dim, int32_t n_ranks);
/* step_size_chain_out [C] (every entry = initial_step_size: the array the transition kernels read as per-chain step
 * sizes), imm_out [D] = ones (also installed as the handle's diagonal metric). */
int bjx_adapt_shared_init(bjx_handle_t h, float* state, float initial_step_size, float* step_size_chain_out, float* imm_out);
/* One warm-up step after the transition: block statistics of (q, acceptance_rate) -> all-gather -> merge, dual
 * averaging, window bookkeeping (stage: 0 fast / 1 slow; window_end: last step of a slow window: imm rewritten,
 * accumulator reset, dual averaging re-initialised, the handle's metric re-installed).  step_size_chain [C] is
 * refilled with the new step size.  eps_history (nullable, device): the step size of warm-up step t lands in [t].
 * Fully asynchronous on the handle's stream. */
int bjx_adapt_shared_update(bjx_handle_t h, void* nccl_comm, int32_t n_ranks, float* state, const float* q,
                            const float* acceptance_rate, int32_t stage, int32_t window_end, float target_acceptance,
                            float* step_size_chain, float* imm, float* eps_history);
/* The whole shared warm-up as one call (staged_adaptation.py:906-966): for t < num_steps one in-place transition with step
 * key split(rng_key, num_steps)[t] (NUTS when max_num_doublings > 0, else HMC with num_integration_steps) followed by
 * bjx_adapt_shared_update with schedule[t] = stage | window_end << 1 (HOST array, staged_adaptation.py:315-405).
 * state / step_size_chain / imm as initialised by bjx_adapt_shared_init; acceptance_scratch: device float32 [C];
 * steps_scratch (device int32 [C]) + leapfrog_counter (device uint64, caller-zeroed): optional, the executed leapfrogs
 * summed over chains and steps.  Asynchronous: the loop only enqueues. */
int bjx_adapt_shared_run(bjx_handle_t h, void* nccl_comm, int32_t n_ranks, const uint32_t* rng_key, const uint8_t* schedule,
                         int32_t num_steps, float* q, float* logp, float* grad, float* state, float* step_size_chain,
                         float* imm, float target_acceptance, int32_t max_num_doublings, int32_t num_integration_steps,
                         float* eps_history, float* acceptance_scratch, int32_t* steps_scratch,
                         unsigned long long* leapfrog_counter);
/* final step size exp(log_step_avg) (staged_adaptation.py:303) into step_size_out [1] (device) */
int bjx_adapt_shared_final(bjx_handle_t h, const float* state, float* step_size_out);

/* ---- ChEES-HMC warm-up (blackjax/adaptation/chees_adaptation.py, mass_matrix_estimation=None; SURVEY 8f item 4) --------------
 * Cross-chain adaptation of the step size (dual averaging on the harmonic mean of the acceptance probabilities) and of the
 * trajectory length (Adam on log T along the ChEES gradient), device resident, two all-gathers of block statistics per
 * step.  The transition is an HMC step with per-chain arrays the update rewrites: step_size_chain [C] (one value) and
 * steps_chain int32 [C] = ceil(jitter(i) * T / eps) with the base-2 Halton jitter (dynamic_hmc.py:205-215); pass the
 * latter to bjx_set_integration_steps and request proposal_position / proposal_momentum in bjx_info. */
int64_t bjx_chees_state_floats(int32_t n_chains_local, int32_t dim, int32_t n_ranks);
int bjx_chees_init(bjx_handle_t h, float* state, float step_size, int32_t max_bits, float jitter_amount,
                   float* step_size_chain_out, int32_t* steps_chain_out);
/* one warm-up step after the transition; optimiser = Adam(learning_rate, b1, b2, eps 1e-8); history (nullable, device
 * [num_steps, 4]) receives (step_size, trajectory_length, next step count, ChEES gradient) */
int bjx_chees_update(bjx_handle_t h, void* nccl_comm, int32_t n_ranks, float* state, const float* initial_position,
                     const float* proposal_position, const float* proposal_momentum, const float* acceptance_rate,
                     const uint8_t* is_divergent, float learning_rate, float b1, float b2, float target_acceptance,
                     float decay_rate, int32_t max_leapfrog_steps, float* step_size_chain, int32_t* steps_chain, float* history);
/* out2 (HOST, 2 floats): step_size = exp(log_step_size_moving_average), num_leapfrog_steps = exp(log T_ma - log eps_ma);
 * synchronises the stream */
int bjx_chees_final(bjx_handle_t h, const float* state, float* out2_host);

/* ---- diagnostics on a device-resident history (SURVEY 8f item 3) ---------------------------------------------- */
/* blackjax.diagnostics.potential_scale_reduction (diagnostics.py:39-89): history float32 [num_samples, C, D] as written
 * by bjx_hmc_sample; rhat_out float32 [D]; scratch: at least 2*C*D + 4 + 4*D floats (device). */
int bjx_potential_scale_reduction(bjx_handle_t h, const float* history, int32_t num_samples, float* rhat_out,
                                  float* scratch);

/* blackjax.diagnostics.effective_sample_size (diagnostics.py:159-305; Geyer initial positive + monotone sequences on
 * the chain-averaged autocovariance), same history layout; ess_out float32 [D]; scratch: 8-byte aligned device buffer of
 * at least bjx_ess_scratch_floats(num_samples, C, D) floats.  One chain is allowed (no between-chain term). */
int64_t bjx_ess_scratch_floats(int32_t num_samples, int32_t n_chains, int32_t dim);
int bjx_effective_sample_size(bjx_handle_t h, const float* history, int32_t num_samples, float* ess_out, float* scratch);

#ifdef __cplusplus
}
#endif
#endif /* BJX_H_ */

// C ABI of libbjx.so (include/bjx.h): handle management, argument checking, kernel dispatch and
// the host-driven NUTS doubling loop.  No torch types, no exceptions across the boundary.
#include <algorithm>
#include <dlfcn.h>
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/bjx.h"
#include "bjx_internal.h"
#include "bjx_launch.cuh"
#include "bjx_big.cuh"
#include "bjx_handle.h"

using namespace bjx;

static thread_local std::string g_err;

int bjx_fail(bjx_handle_t h, int code, const std::string& msg) {
  g_err = msg;
  if (h) h->err = msg;
  return code;
}
int bjx_cuda_fail(bjx_handle_t h, cudaError_t e, const char* where) {
  return bjx_fail(h, (int)e, std::string(where) + ": " + cudaGetErrorString(e));
}
static int fail(bjx_handle_t h, int code, const std::string& msg) { return bjx_fail(h, code, msg); }
static int cuda_fail(bjx_handle_t h, cudaError_t e, const char* where) { return bjx_cuda_fail(h, e, where); }

// large-D dense path (bjx_dense.cu)
int bjx_dense_init_state(bjx_handle_t h, const float* q, float* logp_out, float* grad_out);
int bjx_dense_sample_momentum(bjx_handle_t h, const uint32_t* keys, float* p_out, bool split_first);
int bjx_dense_energy(bjx_handle_t h, const float* p, const float* logp, float* e_out);
int bjx_dense_velocity(bjx_handle_t h, const float* p, float* v);
int bjx_dense_leapfrog(bjx_handle_t h, float* q, float* p, float* logp, float* g, float eps, const float* eps_dev, int n);
int bjx_dense_hmc_step(bjx_handle_t h, const uint32_t* keys, const float* q_in, const float* logp_in, const float* g_in,
                       float* q_out, float* logp_out, float* g_out, float eps, const float* eps_dev, int L,
                       const bjx::InfoPtrs& info);
int bjx_dense_nuts_step(bjx_handle_t h, const uint32_t* keys, const float* q_in, const float* logp_in, const float* g_in,
                        float* q_out, float* logp_out, float* g_out, float step_size, const float* step_size_dev,
                        int max_num_doublings, bjx::InfoPtrs info, const float* momentum_override,
                        const uint32_t* key_integrator_override);
static inline bool target_large_dense(bjx_handle_t h) {
  return h->cfg.target.kind == BJX_TARGET_DENSE_GAUSSIAN && h->cfg.dim > 128;
}
static inline bool metric_large_dense(bjx_handle_t h) { return h->metric_kind == BJX_METRIC_DENSE && h->cfg.dim > 128; }
static inline bool use_dense_path(bjx_handle_t h) { return target_large_dense(h) || metric_large_dense(h); }

// CTA-per-chain path for 1024 < dim <= 18432 (bjx_big.cu)
int bjx_big_init_state(bjx_handle_t h, const float* q, float* logp_out, float* grad_out);
int bjx_big_sample_momentum(bjx_handle_t h, const uint32_t* keys, float* p_out);
int bjx_big_energy(bjx_handle_t h, const float* p, const float* logp, float* e_out);
int bjx_big_leapfrog(bjx_handle_t h, float* q, float* p, float* logp, float* g, float eps, const float* eps_dev, int n);
int bjx_big_hmc_step(bjx_handle_t h, const uint32_t* keys, const float* q_in, const float* logp_in, const float* g_in,
                     float* q_out, float* logp_out, float* g_out, float eps, const float* eps_dev, int L,
                     const bjx::InfoPtrs& info);
static inline bool use_big_path(bjx_handle_t h) { return h->sc == SC_BIG && !use_dense_path(h); }
#define BJX_CUDA(call)                                            \
  do {                                                            \
    cudaError_t e_ = (call);                                      \
    if (e_ != cudaSuccess) return cuda_fail(h, e_, #call);        \
  } while (0)
#define BJX_CHECK_LAUNCH(where)                                   \
  do {                                                            \
    cudaError_t e_ = cudaGetLastError();                          \
    if (e_ != cudaSuccess) return cuda_fail(h, e_, where);        \
  } while (0)

// Dense targets and dense metrics stop at 1024 dims: the tensor-core products accumulate in float32 with truncation at
// each of their 3K/16 steps, so their error grows linearly in K and passes the 1e-5 per product stated for the path
// beyond K = 1024 (DESIGN.md section 3).
constexpr int kDenseMaxDim = 1024;
constexpr const char* kDenseLimitMsg =
    "dense targets and dense metrics are built for dim <= 1024 (beyond, the tensor-core products lose float32 accuracy)";

static int validate_target(bjx_handle_t h, const bjx_target_desc& t, int dim) {
  if (t.dim != dim) return fail(h, BJX_E_INVALID, "target.dim != config.dim");
  switch (t.kind) {
    case BJX_TARGET_DIAG_GAUSSIAN:
      if (!t.inv_var) return fail(h, BJX_E_INVALID, "DIAG_GAUSSIAN target needs inv_var");
      break;
    case BJX_TARGET_FUNNEL:
      if (dim < 2) return fail(h, BJX_E_INVALID, "FUNNEL target needs dim >= 2");
      break;
    case BJX_TARGET_DENSE_GAUSSIAN:
      if (!t.precision) return fail(h, BJX_E_INVALID, "DENSE_GAUSSIAN target needs precision");
      if (dim > 128 && dim % 4 != 0) return fail(h, BJX_E_UNSUPPORTED, "DENSE_GAUSSIAN target with dim > 128 needs dim % 4 == 0 (tensor-core GEMM path)");
      if (dim > kDenseMaxDim) return fail(h, BJX_E_UNSUPPORTED, kDenseLimitMsg);
      break;
    case BJX_TARGET_BANANA:
      if (dim != 2) return fail(h, BJX_E_INVALID, "BANANA target needs dim == 2");
      break;
    case BJX_TARGET_HIER_LOGIT:
      if (!t.data_x || !t.data_y || t.n_groups < 1 || dim != 4 + t.n_groups)
        return fail(h, BJX_E_INVALID, "HIER_LOGIT target needs data_x, data_y and dim == 4 + n_groups");
      if (dim <= 1024 || dim % 4 != 0)
        return fail(h, BJX_E_UNSUPPORTED, "HIER_LOGIT target is built for 1024 < dim <= 18432, dim % 4 == 0 (CTA-per-chain kernels)");
      break;
    case BJX_TARGET_USER:
      if (!t.user_plugin) return fail(h, BJX_E_INVALID, "USER target needs user_plugin (bjx_plugin_load)");
      if (t.n_user_params < 0 || (t.n_user_params > 0 && !t.user_params))
        return fail(h, BJX_E_INVALID, "USER target: user_params is NULL but n_user_params > 0");
      {
        auto* pl = static_cast<bjx_plugin_s*>(t.user_plugin);
        if (dim > 1024 && !pl->launch_big)
          return fail(h, BJX_E_UNSUPPORTED, "this USER target's plug-in holds the warp kernels only (dim <= 1024): build it with "
                                            "bjx_user::BigModel for rows beyond");
        if (dim <= 1024 && !pl->launch)
          return fail(h, BJX_E_UNSUPPORTED, "this USER target's plug-in holds the big-row kernels only (dim > 1024)");
      }
      break;
    default:
      return fail(h, BJX_E_INVALID, "unknown target kind");
  }
  return 0;
}

// ---- plug-ins of user-defined targets (include/bjx_user_target.h) ---------------------------------------------------
// what a plug-in must have been built against: the C ABI version and the layout of the launch arguments
extern "C" int bjx_plugin_abi(void) {
  return BJX_VERSION * 100000 + (int)sizeof(bjx::LaunchArgs) + 7 * (int)sizeof(bjx::BigLaunchArgs);
}

extern "C" int bjx_plugin_load(const char* path, void** plugin_out) {
  if (!path || !plugin_out) return fail(nullptr, BJX_E_INVALID, "null argument");
  void* dl = dlopen(path, RTLD_NOW | RTLD_LOCAL);
  if (!dl) return fail(nullptr, BJX_E_INVALID, std::string("bjx_plugin_load: ") + dlerror());
  auto abi = (int (*)(void))dlsym(dl, "bjx_plugin_built_for_abi");
  auto launch = (int (*)(int, int, int, const bjx::LaunchArgs*))dlsym(dl, "bjx_plugin_launch");
  auto launch_big = (int (*)(int, const bjx::BigLaunchArgs*))dlsym(dl, "bjx_plugin_launch_big");
  if (!abi || (!launch && !launch_big)) {
    dlclose(dl);
    return fail(nullptr, BJX_E_INVALID, std::string("bjx_plugin_load: ") + path + " is not a bjx target plug-in");
  }
  if (abi() != bjx_plugin_abi()) {
    dlclose(dl);
    return fail(nullptr, BJX_E_STATE, std::string("bjx_plugin_load: ") + path +
                                          " was built against another version of libbjx's kernels: rebuild it");
  }
  *plugin_out = new bjx_plugin_s{dl, launch, launch_big};  // never unloaded: handles may refer to it until the process ends
  return 0;
}

extern "C" int bjx_version(void) { return BJX_VERSION; }

extern "C" const char* bjx_last_error(bjx_handle_t h) { return h ? h->err.c_str() : g_err.c_str(); }

extern "C" int bjx_create(const bjx_config* cfg, bjx_handle_t* out) {
  bjx_handle_t h = nullptr;
  if (!cfg || !out) return fail(nullptr, BJX_E_INVALID, "null argument");
  if (cfg->n_chains <= 0 || cfg->dim <= 0) return fail(nullptr, BJX_E_INVALID, "n_chains and dim must be positive");
  if (cfg->max_tree_depth < 1 || cfg->max_tree_depth > 30) return fail(nullptr, BJX_E_INVALID, "max_tree_depth must be in [1, 30]");
  const int sc = size_class_for(cfg->dim);
  if (sc == SC_NONE)
    return fail(nullptr, BJX_E_UNSUPPORTED, "dim must be <= 18432 with dim % 4 == 0, or <= 128 otherwise");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess) return cuda_fail(nullptr, e, "cudaGetDeviceCount (no CUDA device: there is no CPU fallback)");
  if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, BJX_E_INVALID, "bad device ordinal");
  e = cudaSetDevice(cfg->device);
  if (e != cudaSuccess) return cuda_fail(nullptr, e, "cudaSetDevice");
  h = new bjx_handle_s();
  h->cfg = *cfg;
  if (!(h->cfg.divergence_threshold > 0.f)) h->cfg.divergence_threshold = 1000.f;
  h->stream = (cudaStream_t)cfg->stream;
  h->sc = sc;
  h->metric_kind = -1;
  h->metric_small_dense = false;
  h->imm = nullptr;
  h->msqrt = nullptr;
  h->msqrt_elems = 0;
  memset(&h->ws, 0, sizeof(h->ws));
  h->ws_block = nullptr;
  h->ws_depth = 0;
  h->h_flag = nullptr;
  h->last_leaf_launches = 0;
  h->last_depth = 0;
  h->dense_block = nullptr;
  h->dense_bytes = 0;
  h->gemm_ws = nullptr;
  h->gemm_ws_bytes = 0;
  for (int m = 0; m < 3; ++m) { h->dense_mat_s[m] = nullptr; h->dense_mat_src[m] = nullptr; h->dense_mat_ver[m] = 0; }
  h->dense_version = 1;
  h->dense_bytes_built = 0;
  h->pool_scratch = nullptr;
  h->dn_block = nullptr;
  h->dn_bytes = 0;
  h->pool_scratch_bytes = 0;
  h->lr_block = nullptr;
  h->lr_k = 0;
  h->dense_streams_ready = false;
  h->dense_stagger_armed = false;
  h->ncoef = 3;
  h->coef[0] = 0.5f; h->coef[1] = 1.0f; h->coef[2] = 0.5f;
  h->general_integrator = false;
  h->key_shared = 0;
  h->steps_dev = nullptr;
  h->ghmc_noise = nullptr;
  h->chain_offset = 0;
  h->sample_keys = nullptr;
  h->sample_keys_cap = 0;
  int rc = validate_target(h, cfg->target, cfg->dim);
  if (rc) {
    g_err = h->err;
    delete h;
    return rc;
  }
  e = cudaMallocHost((void**)&h->h_flag, 64 * sizeof(int));
  if (e != cudaSuccess) {
    delete h;
    return cuda_fail(nullptr, e, "cudaMallocHost");
  }
  *out = h;
  return 0;
}

extern "C" int bjx_destroy(bjx_handle_t h) {
  if (!h) return 0;
  cudaSetDevice(h->cfg.device);
  cudaStreamSynchronize(h->stream);
  if (h->msqrt) cudaFree(h->msqrt);
  if (h->ws_block) cudaFree(h->ws_block);
  if (h->dense_block) cudaFree(h->dense_block);
  if (h->pool_scratch) cudaFree(h->pool_scratch);
  if (h->dn_block) cudaFree(h->dn_block);
  if (h->lr_block) cudaFree(h->lr_block);
  if (h->gemm_ws) cudaFree(h->gemm_ws);
  if (h->sample_keys) cudaFree(h->sample_keys);
  if (h->dense_streams_ready) {
    for (int k = 0; k < 2; ++k) { cudaStreamDestroy(h->dense_stream[k]); cudaEventDestroy(h->dense_join[k]); }
    cudaEventDestroy(h->dense_fork);
    cudaEventDestroy(h->dense_stagger);
  }
  if (h->h_flag) cudaFreeHost(h->h_flag);
  delete h;
  return 0;
}

extern "C" int bjx_set_target(bjx_handle_t h, const bjx_target_desc* t) {
  if (!h || !t) return fail(h, BJX_E_INVALID, "null argument");
  int rc = validate_target(h, *t, h->cfg.dim);
  if (rc) return rc;
  h->cfg.target = *t;
  h->dense_version++;
  return 0;
}

// integrators.py:62-152,321-369: palindromic coefficient table (host array, odd length 3..11)
extern "C" int bjx_set_integrator(bjx_handle_t h, const float* coefficients, int32_t n) {
  if (!h || !coefficients) return fail(h, BJX_E_INVALID, "null argument");
  if (n < 3 || n > 11 || (n % 2) == 0) return fail(h, BJX_E_INVALID, "integrator needs an odd number (3..11) of coefficients");
  for (int i = 0; i < n; ++i)
    if (coefficients[i] != coefficients[n - 1 - i]) return fail(h, BJX_E_INVALID, "integrator coefficients must be palindromic");
  h->ncoef = n;
  for (int i = 0; i < n; ++i) h->coef[i] = coefficients[i];
  h->general_integrator = !(n == 3 && coefficients[0] == 0.5f && coefficients[1] == 1.0f);
  return 0;
}

// Key source of the transition kernels: 0 = `keys` holds one key per chain [C,2]; 1 = `keys` holds ONE step key [2] and
// chain c uses split(step_key, n_global)[chain_offset + c] (util.py:203 / staged_adaptation.py:920 step-major schedule).
extern "C" int bjx_set_key_mode(bjx_handle_t h, int32_t shared_step_key, uint32_t chain_offset) {
  if (!h) return fail(h, BJX_E_INVALID, "null handle");
  h->key_shared = shared_step_key ? 1 : 0;
  h->chain_offset = chain_offset;
  return 0;
}

// Dynamic HMC (blackjax/mcmc/dynamic_hmc.py:109-120): per-chain numbers of integration steps int32 [C] (device) for the
// following bjx_hmc_step / bjx_mhmc_step calls, whose scalar L is then ignored; NULL restores the scalar.
extern "C" int bjx_set_integration_steps(bjx_handle_t h, const int32_t* steps_dev) {
  if (!h) return fail(h, BJX_E_INVALID, "null handle");
  h->steps_dev = steps_dev;
  return 0;
}

// Generalized HMC's slice noise (blackjax/mcmc/ghmc.py:90,172 `noise_fn(key_noise)`): per-chain values float32 [C]
// (device) added to the slice translation of the following bjx_ghmc_step calls; NULL restores the default (0).
extern "C" int bjx_set_ghmc_noise(bjx_handle_t h, const float* noise_dev) {
  if (!h) return fail(h, BJX_E_INVALID, "null handle");
  h->ghmc_noise = noise_dev;
  return 0;
}

extern "C" int bjx_synchronize(bjx_handle_t h) {
  if (!h) return fail(h, BJX_E_INVALID, "null handle");
  BJX_CUDA(cudaSetDevice(h->cfg.device));
  BJX_CUDA(cudaStreamSynchronize(h->stream));
  return 0;
}

extern "C" int bjx_set_metric(bjx_handle_t h, int32_t kind, const float* imm) {
  if (!h || !imm) return fail(h, BJX_E_INVALID, "null argument");
  BJX_CUDA(cudaSetDevice(h->cfg.device));
  const int D = h->cfg.dim, C = h->cfg.n_chains;
  size_t elems;
  if (kind == BJX_METRIC_DIAG) elems = D;
  else if (kind == BJX_METRIC_DIAG_PER_CHAIN) elems = (size_t)C * D;
  else if (kind == BJX_METRIC_DENSE_PER_CHAIN) {
    if (D > 64) return fail(h, BJX_E_UNSUPPORTED, "per-chain dense metrics are built for dim <= 64");
    elems = (size_t)C * D * D;
  } else if (kind == BJX_METRIC_DENSE) {
    if (D > 128 && D % 4 != 0)
      return fail(h, BJX_E_UNSUPPORTED, "dense metric with dim > 128 needs dim % 4 == 0 (tensor-core GEMM path)");
    if (D > kDenseMaxDim) return fail(h, BJX_E_UNSUPPORTED, kDenseLimitMsg);
    elems = (size_t)D * D;
  } else
    return fail(h, BJX_E_INVALID, "The mass matrix has the wrong number of dimensions: expected 1 or 2");  // metrics.py:724-728
  if (elems > h->msqrt_elems) {
    if (h->msqrt) BJX_CUDA(cudaFree(h->msqrt));
    h->msqrt = nullptr;
    BJX_CUDA(cudaMalloc((void**)&h->msqrt, elems * sizeof(float)));
    h->msqrt_elems = elems;
  }
  if (kind == BJX_METRIC_DENSE) {
    // metrics.py:712-715: L = chol(M^-1) (lower); mass_matrix_sqrt = solve_triangular(L, I, lower, trans) = L^-T
    std::vector<float> a((size_t)D * D);
    BJX_CUDA(cudaMemcpyAsync(a.data(), imm, a.size() * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    BJX_CUDA(cudaStreamSynchronize(h->stream));
    std::vector<double> L((size_t)D * D, 0.0), Li((size_t)D * D, 0.0);
    for (int i = 0; i < D; ++i)
      for (int j = 0; j <= i; ++j) {
        double s = a[(size_t)i * D + j];
        for (int k = 0; k < j; ++k) s -= L[(size_t)i * D + k] * L[(size_t)j * D + k];
        if (i == j) {
          if (!(s > 0.0)) return fail(h, BJX_E_INVALID, "inverse mass matrix is not positive definite");
          L[(size_t)i * D + i] = sqrt(s);
        } else
          L[(size_t)i * D + j] = s / L[(size_t)j * D + j];
      }
    for (int c = 0; c < D; ++c) {  // Li = L^-1 by forward substitution, column c
      for (int i = c; i < D; ++i) {
        double s = (i == c) ? 1.0 : 0.0;
        for (int k = c; k < i; ++k) s -= L[(size_t)i * D + k] * Li[(size_t)k * D + c];
        Li[(size_t)i * D + c] = s / L[(size_t)i * D + i];
      }
    }
    std::vector<float> m((size_t)D * D);
    for (int i = 0; i < D; ++i)
      for (int j = 0; j < D; ++j) m[(size_t)i * D + j] = (float)Li[(size_t)j * D + i];  // (L^-1)^T
    BJX_CUDA(cudaMemcpyAsync(h->msqrt, m.data(), m.size() * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    BJX_CUDA(cudaStreamSynchronize(h->stream));
  } else if (kind == BJX_METRIC_DENSE_PER_CHAIN) {
    launch_chol_linv_t(C, D, imm, h->msqrt, h->stream);  // L^-T per chain on the device (float64)
    BJX_CHECK_LAUNCH("k_chol_linv_t");
  } else {
    launch_diag_mass_sqrt(imm, (long long)elems, h->msqrt, h->stream);
    BJX_CHECK_LAUNCH("k_diag_mass_sqrt");
  }
  h->dense_version++;
  h->metric_kind = kind;
  h->metric_small_dense = ((kind == BJX_METRIC_DENSE) && D <= 128) || kind == BJX_METRIC_DENSE_PER_CHAIN;
  h->imm = imm;
  return 0;
}

static __global__ void k_low_rank_prepare(int D, int k, const float* __restrict__ sigma, const float* __restrict__ lam,
                                          float* __restrict__ sg, float* __restrict__ isg, float* __restrict__ lm1,
                                          float* __restrict__ islm1) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < D) {
    sg[i] = sigma[i];
    isg[i] = 1.0f / sigma[i];                       // inv_sigma (metrics.py:384)
  }
  if (i < k) {
    lm1[i] = lam[i] - 1.0f;
    islm1[i] = 1.0f / sqrtf(lam[i]) - 1.0f;         // inv_sqrt_lam - 1 (metrics.py:385-386, :141)
  }
}

extern "C" int bjx_set_metric_low_rank(bjx_handle_t h, const float* sigma, const float* U, const float* lam, int32_t rank) {
  if (!h || !sigma || !U || !lam) return fail(h, BJX_E_INVALID, "null argument");
  if (rank < 1 || rank > kMaxLowRank) return fail(h, BJX_E_UNSUPPORTED, "low-rank metric: 1 <= rank <= 16");
  const int D = h->cfg.dim;
  if (h->sc == SC_BIG || h->sc == SC_V8 || h->sc == SC_NONE || use_dense_path(h))
    return fail(h, BJX_E_UNSUPPORTED, "low-rank metric is built for the warp kernels with dim <= 512 (dim % 4 == 0 above 128)");
  BJX_CUDA(cudaSetDevice(h->cfg.device));
  const size_t need = ((size_t)D * rank + 2 * (size_t)D + 2 * (size_t)rank) * sizeof(float);
  if (h->lr_block) BJX_CUDA(cudaFree(h->lr_block));
  h->lr_block = nullptr;
  BJX_CUDA(cudaMalloc((void**)&h->lr_block, need));
  float* Ud = h->lr_block;
  float* sg = Ud + (size_t)D * rank;
  BJX_CUDA(cudaMemcpyAsync(Ud, U, (size_t)D * rank * sizeof(float), cudaMemcpyDeviceToDevice, h->stream));
  k_low_rank_prepare<<<(D + 255) / 256, 256, 0, h->stream>>>(D, rank, sigma, lam, sg, sg + D, sg + 2 * D, sg + 2 * D + rank);
  BJX_CHECK_LAUNCH("k_low_rank_prepare");
  h->lr_k = rank;
  h->metric_kind = BJX_METRIC_LOW_RANK;
  h->metric_small_dense = false;
  h->imm = sg;      // (diagonal scaling, for completeness; the low-rank kernels read the lr_* arrays)
  h->dense_version++;
  return 0;
}

extern "C" int bjx_get_mass_matrix_sqrt(bjx_handle_t h, const float** out) {
  if (!h || !out) return fail(h, BJX_E_INVALID, "null argument");
  if (h->metric_kind < 0) return fail(h, BJX_E_STATE, "metric not set");
  *out = h->msqrt;
  return 0;
}

static Params make_params(bjx_handle_t h, float eps, const float* eps_dev) {
  Params P;
  P.C = h->cfg.n_chains;
  P.D = h->cfg.dim;
  P.inv_var = h->cfg.target.inv_var;
  P.mean = h->cfg.target.mean;
  P.prec = h->cfg.target.precision;
  P.logp_offset = h->cfg.target.logp_offset;
  P.user = h->cfg.target.user_params;
  P.n_user = h->cfg.target.n_user_params;
  P.imm = h->imm;
  P.imm_stride = (h->metric_kind == BJX_METRIC_DIAG_PER_CHAIN) ? h->cfg.dim
                 : (h->metric_kind == BJX_METRIC_DENSE_PER_CHAIN) ? (long long)h->cfg.dim * h->cfg.dim : 0;
  P.imm_group = 1;
  P.msqrt = h->msqrt;
  P.lr_k = (h->metric_kind == BJX_METRIC_LOW_RANK) ? h->lr_k : 0;
  if (P.lr_k > 0) {
    const size_t D = h->cfg.dim, k = h->lr_k;
    P.lr_U = h->lr_block;
    P.lr_sigma = h->lr_block + D * k;
    P.lr_inv_sigma = P.lr_sigma + D;
    P.lr_lam_m1 = P.lr_inv_sigma + D;
    P.lr_isl_m1 = P.lr_lam_m1 + k;
  } else {
    P.lr_U = P.lr_sigma = P.lr_inv_sigma = P.lr_lam_m1 = P.lr_isl_m1 = nullptr;
  }
  P.eps = eps;
  P.eps_dev = eps_dev;
  P.div_thr = h->cfg.divergence_threshold;
  P.key_shared = h->key_shared;
  P.chain_offset = h->chain_offset;
  P.steps_dev = h->steps_dev;
  P.ncoef = h->ncoef;
  for (int i = 0; i < 11; ++i) P.coef[i] = i < h->ncoef ? h->coef[i] : 0.f;
  return P;
}

static int dispatch(bjx_handle_t h, int kernel_id, bool target_dependent, LaunchArgs& a) {
  a.stream = h->stream;
  a.general_integrator = h->general_integrator;
  const bool dm = h->metric_small_dense || h->metric_kind == BJX_METRIC_LOW_RANK;
  int rc;
  const int tk = target_dependent ? h->cfg.target.kind : (int)BJX_TARGET_FUNNEL;
  switch (tk) {
    case BJX_TARGET_DIAG_GAUSSIAN: rc = Launcher<TK_DIAG>::launch(kernel_id, h->sc, dm, a); break;
    case BJX_TARGET_FUNNEL: rc = Launcher<TK_FUNNEL>::launch(kernel_id, h->sc, dm, a); break;
    case BJX_TARGET_DENSE_GAUSSIAN: rc = Launcher<TK_DENSE>::launch(kernel_id, h->sc, dm, a); break;
    case BJX_TARGET_BANANA: rc = Launcher<TK_BANANA>::launch(kernel_id, h->sc, dm, a); break;
    case BJX_TARGET_USER:
      if (!static_cast<bjx_plugin_s*>(h->cfg.target.user_plugin)->launch) { rc = -2; break; }
      rc = static_cast<bjx_plugin_s*>(h->cfg.target.user_plugin)->launch(kernel_id, h->sc, dm ? 1 : 0, &a);
      if (rc > 0) return cuda_fail(h, (cudaError_t)rc, "plug-in kernel launch");
      break;
    default: rc = -2;
  }
  if (rc) return fail(h, BJX_E_UNSUPPORTED, "kernel variant not built for this (target, dim, metric, integrator) combination");
  BJX_CHECK_LAUNCH("kernel launch");
  return 0;
}

static int check_ready(bjx_handle_t h, bool need_metric, const void* const* ptrs, int n) {
  if (!h) return fail(h, BJX_E_INVALID, "null handle");
  if (need_metric && h->metric_kind < 0) return fail(h, BJX_E_STATE, "metric not set: call bjx_set_metric first");
  for (int i = 0; i < n; ++i) {
    if (!ptrs[i]) return fail(h, BJX_E_INVALID, "null array argument");
    if (size_class_is_vec(h->sc) && ((uintptr_t)ptrs[i] & 15u)) return fail(h, BJX_E_INVALID, "state arrays must be 16-byte aligned");
  }
  cudaError_t e = cudaSetDevice(h->cfg.device);
  if (e != cudaSuccess) return cuda_fail(h, e, "cudaSetDevice");
  return 0;
}

extern "C" int bjx_init_state(bjx_handle_t h, const float* q, float* logp_out, float* grad_out) {
  const void* ptrs[] = {q, grad_out};
  int rc = check_ready(h, false, ptrs, 2);
  if (rc) return rc;
  if (!logp_out) return fail(h, BJX_E_INVALID, "null array argument");
  if (target_large_dense(h)) return bjx_dense_init_state(h, q, logp_out, grad_out);
  if (h->sc == SC_BIG) return bjx_big_init_state(h, q, logp_out, grad_out);
  LaunchArgs a{};
  a.P = make_params(h, 0.f, nullptr);
  a.q_in = q;
  a.logp_out = logp_out;
  a.g_out = grad_out;
  // k_init_state never reads the metric: route through the non-dense-metric variant unless only dm is built
  return dispatch(h, K_INIT, true, a);
}

extern "C" int bjx_sample_momentum(bjx_handle_t h, const uint32_t* keys, float* p_out) {
  const void* ptrs[] = {p_out};
  int rc = check_ready(h, true, ptrs, 1);
  if (rc) return rc;
  if (!keys) return fail(h, BJX_E_INVALID, "null keys");
  if (metric_large_dense(h)) return bjx_dense_sample_momentum(h, keys, p_out, false);
  if (h->sc == SC_BIG) return bjx_big_sample_momentum(h, keys, p_out);
  LaunchArgs a{};
  a.P = make_params(h, 0.f, nullptr);
  a.keys = keys;
  a.p_io = p_out;
  return dispatch(h, K_MOMENTUM, false, a);
}

extern "C" int bjx_leapfrog(bjx_handle_t h, float* q, float* p, float* logp, float* grad, float step_size,
                            const float* step_size_dev, int32_t n_steps) {
  const void* ptrs[] = {q, p, grad};
  int rc = check_ready(h, true, ptrs, 3);
  if (rc) return rc;
  if (!logp || n_steps < 0) return fail(h, BJX_E_INVALID, "bad argument");
  if ((use_dense_path(h) || use_big_path(h)) && h->general_integrator)
    return fail(h, BJX_E_UNSUPPORTED, "only velocity Verlet is built for dim > 1024 / the tensor-core dense path");
  if (use_dense_path(h)) return bjx_dense_leapfrog(h, q, p, logp, grad, step_size, step_size_dev, n_steps);
  if (use_big_path(h)) return bjx_big_leapfrog(h, q, p, logp, grad, step_size, step_size_dev, n_steps);
  LaunchArgs a{};
  a.P = make_params(h, step_size, step_size_dev);
  a.q_out = q;
  a.p_io = p;
  a.logp_out = logp;
  a.g_out = grad;
  a.n = n_steps;
  return dispatch(h, K_LEAPFROG, true, a);
}

extern "C" int bjx_metric_velocity(bjx_handle_t h, const float* p, float* v_out) {
  const void* ptrs[] = {p, v_out};
  int rc = check_ready(h, true, ptrs, 2);
  if (rc) return rc;
  if (h->cfg.dim > 128) {
    if (h->cfg.dim % 4) return fail(h, BJX_E_UNSUPPORTED, "bjx_metric_velocity needs dim % 4 == 0 for dim > 128");
    return bjx_dense_velocity(h, p, v_out);
  }
  return fail(h, BJX_E_UNSUPPORTED, "bjx_metric_velocity is built for dim > 128 (use bjx_energy / bjx_leapfrog below)");
}

extern "C" int bjx_energy(bjx_handle_t h, const float* p, const float* logp, float* energy_out) {
  const void* ptrs[] = {p};
  int rc = check_ready(h, true, ptrs, 1);
  if (rc) return rc;
  if (!logp || !energy_out) return fail(h, BJX_E_INVALID, "null array argument");
  if (metric_large_dense(h)) return bjx_dense_energy(h, p, logp, energy_out);
  if (h->sc == SC_BIG) return bjx_big_energy(h, p, logp, energy_out);
  LaunchArgs a{};
  a.P = make_params(h, 0.f, nullptr);
  a.p_io = const_cast<float*>(p);
  a.logp_in = logp;
  a.e_out = energy_out;
  return dispatch(h, K_ENERGY, false, a);
}

extern "C" int bjx_is_turning(bjx_handle_t h, const float* pl, const float* pr, const float* ps, uint8_t* out) {
  const void* ptrs[] = {pl, pr, ps};
  int rc = check_ready(h, true, ptrs, 3);
  if (rc) return rc;
  if (!out) return fail(h, BJX_E_INVALID, "null array argument");
  if (metric_large_dense(h)) return fail(h, BJX_E_UNSUPPORTED, "U-turn test with a dense metric needs dim <= 128");
  if (h->sc == SC_BIG) return fail(h, BJX_E_UNSUPPORTED, "U-turn test / NUTS are built for dim <= 1024");
  LaunchArgs a{};
  a.P = make_params(h, 0.f, nullptr);
  a.pl = pl;
  a.pr = pr;
  a.ps = ps;
  a.out_u8 = out;
  return dispatch(h, K_TURNING, false, a);
}

static InfoPtrs make_info(const bjx_info* info) {
  InfoPtrs ip{};
  if (info) {
    ip.acceptance_rate = info->acceptance_rate;
    ip.is_accepted = info->is_accepted;
    ip.is_divergent = info->is_divergent;
    ip.is_turning = info->is_turning;
    ip.energy = info->energy;
    ip.num_integration_steps = info->num_integration_steps;
    ip.num_trajectory_expansions = info->num_trajectory_expansions;
    ip.momentum = info->momentum;
    ip.proposal_position = info->proposal_position;
    ip.proposal_momentum = info->proposal_momentum;
  }
  return ip;
}

extern "C" int bjx_hmc_step(bjx_handle_t h, const uint32_t* keys, const float* q_in, const float* logp_in,
                            const float* grad_in, float* q_out, float* logp_out, float* grad_out, float step_size,
                            const float* step_size_dev, int32_t L, const bjx_info* info) {
  const void* ptrs[] = {q_in, grad_in, q_out, grad_out};
  int rc = check_ready(h, true, ptrs, 4);
  if (rc) return rc;
  if (!keys || !logp_in || !logp_out || L < 0) return fail(h, BJX_E_INVALID, "bad argument");
  if ((q_in == q_out) != (grad_in == grad_out) || (q_in == q_out) != (logp_in == logp_out))
    return fail(h, BJX_E_INVALID, "in-place call must alias all of (q, logp, grad)");
  if ((use_dense_path(h) || use_big_path(h)) && h->general_integrator)
    return fail(h, BJX_E_UNSUPPORTED, "only velocity Verlet is built for dim > 1024 / the tensor-core dense path");
  if ((use_dense_path(h) || use_big_path(h)) && h->steps_dev)
    return fail(h, BJX_E_UNSUPPORTED, "per-chain integration steps need dim <= 1024 and the row-resident kernels");
  if (use_dense_path(h))
    return bjx_dense_hmc_step(h, keys, q_in, logp_in, grad_in, q_out, logp_out, grad_out, step_size, step_size_dev, L,
                              make_info(info));
  if (use_big_path(h))
    return bjx_big_hmc_step(h, keys, q_in, logp_in, grad_in, q_out, logp_out, grad_out, step_size, step_size_dev, L,
                            make_info(info));
  LaunchArgs a{};
  a.P = make_params(h, step_size, step_size_dev);
  a.keys = keys;
  a.q_in = q_in;
  a.logp_in = logp_in;
  a.g_in = grad_in;
  a.q_out = q_out;
  a.logp_out = logp_out;
  a.g_out = grad_out;
  a.n = L;
  a.info = make_info(info);
  return dispatch(h, K_HMC, true, a);
}

// ghmc.build_kernel().kernel (ghmc.py:118-189), in place on the persistent (q, p, logp, grad, slice)
extern "C" int bjx_ghmc_step(bjx_handle_t h, const uint32_t* keys, float* q, float* p, float* logp, float* grad, float* slice,
                             float step_size, const float* step_size_dev, float alpha, const float* alpha_dev, float delta,
                             const float* delta_dev, const float* imm_rows, const float* msqrt_rows, int32_t chains_per_group,
                             int32_t skip_begin, int32_t skip_end, const bjx_info* info) {
  const void* ptrs[] = {q, grad, p};
  int rc = check_ready(h, true, ptrs, 3);
  if (rc) return rc;
  if (!keys || !logp || !slice) return fail(h, BJX_E_INVALID, "bad argument");
  if (use_dense_path(h) || use_big_path(h))
    return fail(h, BJX_E_UNSUPPORTED, "generalized HMC is built for dim <= 1024 (dense metrics: dim <= 128)");
  if ((imm_rows != nullptr) != (msqrt_rows != nullptr) || chains_per_group < 1)
    return fail(h, BJX_E_INVALID, "imm_rows and msqrt_rows come together; chains_per_group >= 1");
  if (imm_rows && (h->metric_small_dense || h->metric_kind == BJX_METRIC_LOW_RANK))
    return fail(h, BJX_E_INVALID, "per-row momentum scales need a diagonal metric on the handle");
  LaunchArgs a{};
  a.P = make_params(h, step_size, step_size_dev);
  if (imm_rows) {  // MEADS: one inverse-mass row per fold (meads_adaptation.py:587-606)
    a.P.imm = imm_rows;
    a.P.msqrt = msqrt_rows;
    a.P.imm_stride = h->cfg.dim;
    a.P.imm_group = chains_per_group;
  }
  a.keys = keys;
  a.q_out = q; a.logp_out = logp; a.g_out = grad;
  a.ghmc.p_io = p;
  a.ghmc.slice_io = slice;
  a.ghmc.alpha = alpha; a.ghmc.alpha_dev = alpha_dev;
  a.ghmc.delta = delta; a.ghmc.delta_dev = delta_dev;
  a.ghmc.param_group = chains_per_group;
  a.ghmc.skip_begin = skip_begin; a.ghmc.skip_end = skip_end;
  a.ghmc.noise_dev = h->ghmc_noise;
  a.info = make_info(info);
  return dispatch(h, K_GHMC, true, a);
}

// hmc.build_kernel(build_proposal=multinomial_hmc_proposal) / blackjax.mhmc (hmc.py:181-248, __init__.py:145-151)
extern "C" int bjx_mhmc_step(bjx_handle_t h, const uint32_t* keys, const float* q_in, const float* logp_in,
                             const float* grad_in, float* q_out, float* logp_out, float* grad_out, float step_size,
                             const float* step_size_dev, int32_t L, const bjx_info* info) {
  const void* ptrs[] = {q_in, grad_in, q_out, grad_out};
  int rc = check_ready(h, true, ptrs, 4);
  if (rc) return rc;
  if (!keys || !logp_in || !logp_out || L < 1) return fail(h, BJX_E_INVALID, "bad argument");
  if ((q_in == q_out) != (grad_in == grad_out) || (q_in == q_out) != (logp_in == logp_out))
    return fail(h, BJX_E_INVALID, "in-place call must alias all of (q, logp, grad)");
  if (use_dense_path(h) || h->sc == SC_BIG)
    return fail(h, BJX_E_UNSUPPORTED, "multinomial HMC is built for dim <= 1024 (dense metrics: dim <= 128)");
  LaunchArgs a{};
  a.P = make_params(h, step_size, step_size_dev);
  a.keys = keys;
  a.q_in = q_in; a.logp_in = logp_in; a.g_in = grad_in;
  a.q_out = q_out; a.logp_out = logp_out; a.g_out = grad_out;
  a.n = L;
  a.info = make_info(info);
  return dispatch(h, K_MHMC, true, a);
}

// run_inference_algorithm (blackjax/util.py:150-213) for HMC / multinomial HMC, natively: keys = split(rng_key,
// num_steps) (util.py:203) on the device, then num_steps transitions enqueued back to back with NO host
// synchronisation; per-chain keys come from the step key inside the kernel (bjx_set_key_mode's chain_offset is
// honoured).  history (optional) receives the positions after every `thin`-th transition.
extern "C" int bjx_hmc_sample(bjx_handle_t h, const uint32_t* rng_key, float* q, float* logp, float* grad, float step_size,
                              const float* step_size_dev, int32_t L, int32_t num_steps, int32_t multinomial,
                              float* history, int32_t thin, float* acceptance_history) {
  if (!h || !rng_key || num_steps < 0 || thin < 1) return fail(h, BJX_E_INVALID, "bad argument");
  BJX_CUDA(cudaSetDevice(h->cfg.device));
  if (num_steps == 0) return 0;
  if ((size_t)num_steps > h->sample_keys_cap) {
    if (h->sample_keys) BJX_CUDA(cudaFree(h->sample_keys));
    h->sample_keys = nullptr;
    BJX_CUDA(cudaMalloc((void**)&h->sample_keys, (size_t)num_steps * 2 * sizeof(uint32_t)));
    h->sample_keys_cap = (size_t)num_steps;
  }
  launch_prng_split(rng_key, 1, num_steps, h->sample_keys, h->stream);
  BJX_CHECK_LAUNCH("k_prng_split");
  const int saved_mode = h->key_shared;
  h->key_shared = 1;
  const size_t row_bytes = (size_t)h->cfg.n_chains * h->cfg.dim * sizeof(float);
  int rc = 0;
  for (int t = 0; t < num_steps && rc == 0; ++t) {
    bjx_info info{};
    info.acceptance_rate = acceptance_history ? acceptance_history + (size_t)t * h->cfg.n_chains : nullptr;
    const uint32_t* key_t = h->sample_keys + 2 * (size_t)t;
    rc = multinomial ? bjx_mhmc_step(h, key_t, q, logp, grad, q, logp, grad, step_size, step_size_dev, L, &info)
                     : bjx_hmc_step(h, key_t, q, logp, grad, q, logp, grad, step_size, step_size_dev, L, &info);
    if (rc == 0 && history && ((t + 1) % thin) == 0) {
      cudaError_t e = cudaMemcpyAsync(history + (size_t)((t + 1) / thin - 1) * h->cfg.n_chains * h->cfg.dim, q, row_bytes,
                                      cudaMemcpyDeviceToDevice, h->stream);
      if (e != cudaSuccess) rc = cuda_fail(h, e, "cudaMemcpyAsync(history)");
    }
  }
  h->key_shared = saved_mode;
  return rc;
}

// ---- NUTS workspace -------------------------------------------------------------------------------------
static int ensure_ws(bjx_handle_t h) {
  const int depth = h->cfg.max_tree_depth;
  if (h->ws_block && h->ws_depth == depth) return 0;
  if (h->ws_block) {
    BJX_CUDA(cudaFree(h->ws_block));
    h->ws_block = nullptr;
  }
  const size_t C = h->cfg.n_chains, D = h->cfg.dim;
  const size_t row = ((C * D * sizeof(float)) + 255) & ~(size_t)255;
  const size_t vec = ((C * sizeof(float)) + 255) & ~(size_t)255;
  const size_t key = ((C * 2 * sizeof(uint32_t)) + 255) & ~(size_t)255;
  const size_t ckpt = ((C * depth * D * sizeof(float)) + 255) & ~(size_t)255;
  const size_t n_counters = 64;
  const size_t total = 9 * row + 2 * ckpt + 12 * vec + key + n_counters * sizeof(int) + 256;
  BJX_CUDA(cudaMalloc(&h->ws_block, total));
  BJX_CUDA(cudaMemsetAsync(h->ws_block, 0, total, h->stream));
  char* p = (char*)h->ws_block;
  auto takef = [&](size_t bytes) { float* r = (float*)p; p += bytes; return r; };
  NutsWs& w = h->ws;
  w.left_q = takef(row); w.left_p = takef(row); w.left_g = takef(row);
  w.right_q = takef(row); w.right_p = takef(row); w.right_g = takef(row);
  w.psum = takef(row); w.sub_prop_q = takef(row); w.sub_prop_g = takef(row);
  w.ckpt_p = takef(ckpt); w.ckpt_sum = takef(ckpt);
  w.left_logp = takef(vec); w.right_logp = takef(vec); w.h0 = takef(vec);
  w.prop_energy = takef(vec); w.prop_weight = takef(vec); w.prop_slpa = takef(vec);
  w.n_states = (int*)takef(vec); w.step = (int*)takef(vec);
  w.is_div = (uint8_t*)takef(vec); w.is_turn = (uint8_t*)takef(vec);
  w.list_a = (int*)takef(vec); w.list_b = (int*)takef(vec);
  w.key_int = (uint32_t*)takef(key);
  w.counters = (int*)p;
  w.max_depth = depth;
  h->ws_depth = depth;
  return 0;
}

int bjx_ensure_nuts_ws(bjx_handle_t h) { return ensure_ws(h); }

extern "C" int bjx_nuts_step(bjx_handle_t h, const uint32_t* keys, const float* q_in, const float* logp_in,
                             const float* grad_in, float* q_out, float* logp_out, float* grad_out, float step_size,
                             const float* step_size_dev, int32_t max_num_doublings, const bjx_info* info,
                             const float* momentum_override, const uint32_t* key_integrator_override) {
  const void* ptrs[] = {q_in, grad_in, q_out, grad_out};
  int rc = check_ready(h, true, ptrs, 4);
  if (rc) return rc;
  if (!logp_in || !logp_out) return fail(h, BJX_E_INVALID, "null array argument");
  if ((momentum_override == nullptr) != (key_integrator_override == nullptr))
    return fail(h, BJX_E_INVALID, "momentum_override and key_integrator_override go together");
  if (!keys && !key_integrator_override) return fail(h, BJX_E_INVALID, "null keys");
  if (max_num_doublings < 0 || max_num_doublings > h->cfg.max_tree_depth)
    return fail(h, BJX_E_INVALID, "max_num_doublings exceeds the handle's max_tree_depth");
  if ((q_in == q_out) != (grad_in == grad_out) || (q_in == q_out) != (logp_in == logp_out))
    return fail(h, BJX_E_INVALID, "in-place call must alias all of (q, logp, grad)");
  if (h->sc == SC_BIG && !use_dense_path(h)) return fail(h, BJX_E_UNSUPPORTED, "NUTS is built for dim <= 1024");
  if (use_dense_path(h) && h->general_integrator)
    return fail(h, BJX_E_UNSUPPORTED, "only velocity Verlet is built for the tensor-core dense path");
  auto endpoint_info = [&]() -> int {
    if (info) {
      const size_t bytes = (size_t)h->cfg.n_chains * h->cfg.dim * sizeof(float);
      if (info->left_position) BJX_CUDA(cudaMemcpyAsync(info->left_position, h->ws.left_q, bytes, cudaMemcpyDeviceToDevice, h->stream));
      if (info->left_momentum) BJX_CUDA(cudaMemcpyAsync(info->left_momentum, h->ws.left_p, bytes, cudaMemcpyDeviceToDevice, h->stream));
      if (info->right_position) BJX_CUDA(cudaMemcpyAsync(info->right_position, h->ws.right_q, bytes, cudaMemcpyDeviceToDevice, h->stream));
      if (info->right_momentum) BJX_CUDA(cudaMemcpyAsync(info->right_momentum, h->ws.right_p, bytes, cudaMemcpyDeviceToDevice, h->stream));
    }
    return 0;
  };
  if (use_dense_path(h)) {  // dense metric / dense target beyond 128 dims: lock-step leaves on the tensor-core products
    rc = bjx_dense_nuts_step(h, keys, q_in, logp_in, grad_in, q_out, logp_out, grad_out, step_size, step_size_dev,
                             max_num_doublings, make_info(info), momentum_override, key_integrator_override);
    return rc ? rc : endpoint_info();
  }
  rc = ensure_ws(h);
  if (rc) return rc;
  const int C = h->cfg.n_chains;
  BJX_CUDA(cudaMemsetAsync(h->ws.counters, 0, 64 * sizeof(int), h->stream));

  LaunchArgs a{};
  a.P = make_params(h, step_size, step_size_dev);
  a.ws = h->ws;
  a.keys = keys;
  a.q_in = q_in; a.logp_in = logp_in; a.g_in = grad_in;
  a.q_out = q_out; a.logp_out = logp_out; a.g_out = grad_out;
  a.mom_override = momentum_override;
  a.keyint_override = key_integrator_override;
  a.mom_out = info ? info->momentum : nullptr;
  a.n = max_num_doublings;
  rc = dispatch(h, K_NUTS_INIT, false, a);
  if (rc) return rc;

  // Tree doubling (trajectory.py:616-725) driven from the host WITHOUT a host round trip.  The first kFusedDoublings
  // doublings run in ONE launch over all chains (every chain needs them and their cost is the fixed per-doubling row
  // traffic) and compact the chains that keep expanding into list_a; every further doubling is one launch over the
  // compacted list of the chains still expanding (ping-pong lists), whose length is read on the device from
  // counters[launch]: a fixed grid strides over the list, so a doubling that nobody needs costs one empty launch.
  // Chains never interact, so nothing forces them through the tree in lock step.
  const int kFusedDoublings = 4;  // (the kernel's lane-parallel key schedule handles up to 10 doublings per launch)
  const size_t ckpt_bytes = sizeof(float) * kWarpsPerBlock * 2 * (size_t)h->cfg.max_tree_depth * h->cfg.dim;
  const size_t dm_bytes = (h->metric_small_dense || h->metric_kind == BJX_METRIC_LOW_RANK ||
                           h->cfg.target.kind == BJX_TARGET_DENSE_GAUSSIAN || h->cfg.target.kind == BJX_TARGET_USER)
                              ? sizeof(float) * kWarpsPerBlock * h->cfg.dim : 0;
  a.ckpt_smem = (ckpt_bytes + dm_bytes <= 40 * 1024) ? 1 : 0;  // stay under the 48 KB default dynamic-smem limit
  int64_t launches = 0;
  const int d_fused = max_num_doublings < kFusedDoublings ? max_num_doublings : kFusedDoublings;
  if (max_num_doublings > 0) {
    a.depth = 0;
    a.depth_end = d_fused;
    a.list_in = nullptr;
    a.n_in = C;
    a.n_in_dev = nullptr;
    a.list_out = h->ws.list_a;
    a.counter = h->ws.counters + 1;
    rc = dispatch(h, K_NUTS_DOUBLING, true, a);
    if (rc) return rc;
    ++launches;
  }
  for (int d = d_fused; d < max_num_doublings; ++d) {
    a.depth = d;
    a.depth_end = d + 1;
    a.list_in = (launches & 1) ? h->ws.list_a : h->ws.list_b;
    a.n_in = C;
    a.n_in_dev = h->ws.counters + launches;
    a.list_out = (launches & 1) ? h->ws.list_b : h->ws.list_a;
    a.counter = h->ws.counters + launches + 1;
    rc = dispatch(h, K_NUTS_DOUBLING, true, a);
    if (rc) return rc;
    ++launches;
  }
  k_nuts_finish<<<(C + 255) / 256, 256, 0, h->stream>>>(C, h->ws, make_info(info));
  BJX_CHECK_LAUNCH("k_nuts_finish");
  rc = endpoint_info();
  if (rc) return rc;
  h->last_leaf_launches = launches;
  h->last_depth = -1;  // known on the device only: bjx_nuts_last_stats reads it back on demand
  return 0;
}

extern "C" int bjx_nuts_last_stats(bjx_handle_t h, int64_t* leaf_launches, int64_t* depth_reached) {
  if (!h) return fail(h, BJX_E_INVALID, "null handle");
  if (leaf_launches) *leaf_launches = h->last_leaf_launches;
  if (depth_reached) {
    if (h->last_depth < 0 && h->ws_block) {  // the one host round trip of the NUTS path, and only on request
      BJX_CUDA(cudaMemcpyAsync(h->h_flag, h->ws.counters + 63, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
      BJX_CUDA(cudaStreamSynchronize(h->stream));
      h->last_depth = h->h_flag[0];
    }
    *depth_reached = h->last_depth;
  }
  return 0;
}

// blackjax.util.run_inference_algorithm (util.py:150-213) for NUTS, run natively: step keys = split(rng_key, num_steps) on
// the device, num_steps in-place transitions enqueued back to back; bjx_nuts_step never waits for the device, so neither
// does this loop.  Optional outputs per step: positions (every thin-th), acceptance rates and tree sizes.
extern "C" int bjx_nuts_sample(bjx_handle_t h, const uint32_t* rng_key, float* q, float* logp, float* grad, float step_size,
                               const float* step_size_dev, int32_t max_num_doublings, int32_t num_steps, float* history,
                               int32_t thin, float* acceptance_history, int32_t* num_integration_steps_history) {
  if (!h || !rng_key || num_steps < 0 || thin < 1) return fail(h, BJX_E_INVALID, "bad argument");
  BJX_CUDA(cudaSetDevice(h->cfg.device));
  if (num_steps == 0) return 0;
  if ((size_t)num_steps > h->sample_keys_cap) {
    if (h->sample_keys) BJX_CUDA(cudaFree(h->sample_keys));
    h->sample_keys = nullptr;
    BJX_CUDA(cudaMalloc((void**)&h->sample_keys, (size_t)num_steps * 2 * sizeof(uint32_t)));
    h->sample_keys_cap = (size_t)num_steps;
  }
  launch_prng_split(rng_key, 1, num_steps, h->sample_keys, h->stream);
  BJX_CHECK_LAUNCH("k_prng_split");
  const int saved_mode = h->key_shared;
  h->key_shared = 1;
  const size_t C = h->cfg.n_chains, row_bytes = C * h->cfg.dim * sizeof(float);
  int rc = 0;
  // Enough transitions to amortise the ragged end: the chains run decoupled, every warp taking whole chains through all
  // num_steps transitions (k_nuts_chains).  BJX_NUTS_DECOUPLED=0 keeps the step-synchronous loop (same results).
  static const bool decoupled_ok = [] { const char* e = getenv("BJX_NUTS_DECOUPLED"); return !(e && e[0] == '0'); }();
  if (decoupled_ok && num_steps >= 4 && max_num_doublings > 0 && !use_dense_path(h)) {  // (the dense path is lock step)
    const void* ptrs[] = {q, grad};
    rc = check_ready(h, true, ptrs, 2);
    if (rc == 0 && !logp) rc = fail(h, BJX_E_INVALID, "null array argument");
    if (rc == 0 && max_num_doublings > h->cfg.max_tree_depth)
      rc = fail(h, BJX_E_INVALID, "max_num_doublings exceeds the handle's max_tree_depth");
    if (rc == 0 && h->sc == SC_BIG) rc = fail(h, BJX_E_UNSUPPORTED, "NUTS is built for dim <= 1024");
    if (rc == 0) rc = ensure_ws(h);
    if (rc == 0) {
      cudaError_t e = cudaMemsetAsync(h->ws.counters, 0, 64 * sizeof(int), h->stream);
      if (e != cudaSuccess) rc = cuda_fail(h, e, "cudaMemsetAsync(counters)");
    }
    if (rc == 0) {
      LaunchArgs a{};
      a.P = make_params(h, step_size, step_size_dev);
      a.ws = h->ws;
      a.q_out = q; a.logp_out = logp; a.g_out = grad;
      const size_t ckpt_bytes = sizeof(float) * kWarpsPerBlock * 2 * (size_t)max_num_doublings * h->cfg.dim;
      const size_t dm_bytes = (h->metric_small_dense || h->metric_kind == BJX_METRIC_LOW_RANK ||
                               h->cfg.target.kind == BJX_TARGET_DENSE_GAUSSIAN || h->cfg.target.kind == BJX_TARGET_USER)
                                  ? sizeof(float) * kWarpsPerBlock * h->cfg.dim : 0;
      a.sample.step_keys = h->sample_keys;
      a.sample.num_steps = num_steps;
      a.sample.max_doublings = max_num_doublings;
      a.sample.ckpt_smem = (ckpt_bytes + dm_bytes <= 40 * 1024) ? 1 : 0;
      a.sample.history = history;
      a.sample.thin = thin;
      a.sample.acceptance_history = acceptance_history;
      a.sample.nint_history = num_integration_steps_history;
      a.sample.leapfrogs = nullptr;
      a.sample.queue = h->ws.counters + 62;
      int sms = 148;
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->cfg.device);
      a.grid_override = sms;  // the launcher multiplies by the CTAs that stay resident per SM
      rc = dispatch(h, K_NUTS_CHAINS, true, a);
      h->last_leaf_launches = 1;
      h->last_depth = -1;
    }
    h->key_shared = saved_mode;
    return rc;
  }
  for (int t = 0; t < num_steps && rc == 0; ++t) {
    bjx_info info{};
    info.acceptance_rate = acceptance_history ? acceptance_history + (size_t)t * C : nullptr;
    info.num_integration_steps = num_integration_steps_history ? num_integration_steps_history + (size_t)t * C : nullptr;
    rc = bjx_nuts_step(h, h->sample_keys + 2 * (size_t)t, q, logp, grad, q, logp, grad, step_size, step_size_dev,
                       max_num_doublings, &info, nullptr, nullptr);
    if (rc == 0 && history && ((t + 1) % thin) == 0) {
      cudaError_t e = cudaMemcpyAsync(history + (size_t)((t + 1) / thin - 1) * C * h->cfg.dim, q, row_bytes,
                                      cudaMemcpyDeviceToDevice, h->stream);
      if (e != cudaSuccess) rc = cuda_fail(h, e, "cudaMemcpyAsync(history)");
    }
  }
  h->key_shared = saved_mode;
  return rc;
}

static __global__ void k_accum_steps(int C, const int* __restrict__ n, unsigned long long* __restrict__ out) {
  unsigned long long a = 0;
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < C; c += gridDim.x * blockDim.x) a += (unsigned long long)n[c];
  for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  if ((threadIdx.x & 31) == 0 && a) atomicAdd(out, a);
}

// window_adaptation(...).run for the shared (one step size, one diagonal metric) recipe, run natively
// (staged_adaptation.py:906-966): per warm-up step one transition (NUTS: max_num_doublings > 0, HMC: num_integration_steps
// > 0) with split(rng_key, num_steps)[t] as the step key, then bjx_adapt_shared_update.  schedule[t] = stage | (window_end
// << 1) (staged_adaptation.py:315-405).  Nothing in the loop waits for the device.
extern "C" int bjx_adapt_shared_run(bjx_handle_t h, void* nccl_comm, int32_t n_ranks, const uint32_t* rng_key,
                                    const uint8_t* schedule, int32_t num_steps, float* q, float* logp, float* grad,
                                    float* state, float* step_size_chain, float* imm, float target_acceptance,
                                    int32_t max_num_doublings, int32_t num_integration_steps, float* eps_history,
                                    float* acceptance_scratch, int32_t* steps_scratch, unsigned long long* leapfrog_counter) {
  if (!h || !rng_key || !schedule || !q || !logp || !grad || !state || !step_size_chain || !imm || !acceptance_scratch || num_steps < 0)
    return fail(h, BJX_E_INVALID, "bad argument");
  if ((max_num_doublings > 0) == (num_integration_steps > 0))
    return fail(h, BJX_E_INVALID, "give max_num_doublings (NUTS) or num_integration_steps (HMC)");
  BJX_CUDA(cudaSetDevice(h->cfg.device));
  if (num_steps == 0) return 0;
  if ((size_t)num_steps > h->sample_keys_cap) {
    if (h->sample_keys) BJX_CUDA(cudaFree(h->sample_keys));
    h->sample_keys = nullptr;
    BJX_CUDA(cudaMalloc((void**)&h->sample_keys, (size_t)num_steps * 2 * sizeof(uint32_t)));
    h->sample_keys_cap = (size_t)num_steps;
  }
  launch_prng_split(rng_key, 1, num_steps, h->sample_keys, h->stream);
  BJX_CHECK_LAUNCH("k_prng_split");
  const int saved_mode = h->key_shared;
  h->key_shared = 1;
  int rc = 0;
  for (int t = 0; t < num_steps && rc == 0; ++t) {
    bjx_info info{};
    info.acceptance_rate = acceptance_scratch;
    info.num_integration_steps = (leapfrog_counter && steps_scratch) ? steps_scratch : nullptr;
    const uint32_t* key_t = h->sample_keys + 2 * (size_t)t;
    rc = max_num_doublings > 0
             ? bjx_nuts_step(h, key_t, q, logp, grad, q, logp, grad, 0.f, step_size_chain, max_num_doublings, &info, nullptr, nullptr)
             : bjx_hmc_step(h, key_t, q, logp, grad, q, logp, grad, 0.f, step_size_chain, num_integration_steps, &info);
    if (rc == 0 && info.num_integration_steps) {  // executed leapfrogs, accumulated on the device (bench.py)
      k_accum_steps<<<148, 256, 0, h->stream>>>(h->cfg.n_chains, steps_scratch, leapfrog_counter);
      BJX_CHECK_LAUNCH("k_accum_steps");
    }
    if (rc == 0)
      rc = bjx_adapt_shared_update(h, nccl_comm, n_ranks, state, q, acceptance_scratch, schedule[t] & 1, (schedule[t] >> 1) & 1,
                                   target_acceptance, step_size_chain, imm, eps_history);
  }
  h->key_shared = saved_mode;
  return rc;
}

// ---- PRNG ----------------------------------------------------------------------------------------------
// h may be NULL: the call then runs on the calling thread's registered stream (bjx_set_default_stream; the legacy
// default stream until one is registered).
static thread_local cudaStream_t t_default_stream = (cudaStream_t)0;
extern "C" int bjx_set_default_stream(void* stream) {
  t_default_stream = (cudaStream_t)stream;
  return 0;
}
#define BJX_PRNG_PROLOGUE()                                                        \
  if (!keys || !out || n_keys < 0) return fail(h, BJX_E_INVALID, "bad argument");  \
  if (h) BJX_CUDA(cudaSetDevice(h->cfg.device));                                   \
  cudaStream_t pstream = h ? h->stream : t_default_stream;

extern "C" int bjx_prng_split(bjx_handle_t h, const uint32_t* keys, int64_t n_keys, int32_t num, uint32_t* out) {
  BJX_PRNG_PROLOGUE();
  if (num < 0) return fail(h, BJX_E_INVALID, "bad argument");
  launch_prng_split(keys, n_keys, num, out, pstream);
  BJX_CHECK_LAUNCH("k_prng_split");
  return 0;
}
extern "C" int bjx_prng_fold_in(bjx_handle_t h, const uint32_t* keys, int64_t n_keys, uint32_t data, uint32_t* out) {
  BJX_PRNG_PROLOGUE();
  launch_prng_fold_in(keys, n_keys, data, out, pstream);
  BJX_CHECK_LAUNCH("k_prng_fold_in");
  return 0;
}
extern "C" int bjx_prng_random_bits(bjx_handle_t h, const uint32_t* keys, int64_t n_keys, int64_t per_key, uint32_t* out) {
  BJX_PRNG_PROLOGUE();
  if (per_key < 0 || per_key > 0xFFFFFFFFll) return fail(h, BJX_E_INVALID, "bad per_key");
  launch_prng_draw(0, keys, n_keys, per_key, out, pstream);
  BJX_CHECK_LAUNCH("k_prng_draw");
  return 0;
}
extern "C" int bjx_prng_uniform(bjx_handle_t h, const uint32_t* keys, int64_t n_keys, int64_t per_key, float* out) {
  BJX_PRNG_PROLOGUE();
  if (per_key < 0 || per_key > 0xFFFFFFFFll) return fail(h, BJX_E_INVALID, "bad per_key");
  launch_prng_draw(1, keys, n_keys, per_key, out, pstream);
  BJX_CHECK_LAUNCH("k_prng_draw");
  return 0;
}
// jax.random.randint(key, shape, minval, maxval) int32 (jax/_src/random.py _randint: two 32-bit draws from split(key),
// combined modulo the span with the 2^32 % span multiplier)
extern "C" int bjx_prng_randint(bjx_handle_t h, const uint32_t* keys, int64_t n_keys, int64_t per_key, int32_t minval,
                                int32_t maxval, int32_t* out) {
  BJX_PRNG_PROLOGUE();
  if (per_key < 0 || per_key > 0xFFFFFFFFll) return fail(h, BJX_E_INVALID, "bad per_key");
  launch_prng_randint(keys, n_keys, per_key, minval, maxval, out, pstream);
  BJX_CHECK_LAUNCH("k_prng_randint");
  return 0;
}
extern "C" int bjx_prng_normal(bjx_handle_t h, const uint32_t* keys, int64_t n_keys, int64_t per_key, float* out) {
  BJX_PRNG_PROLOGUE();
  if (per_key < 0 || per_key > 0xFFFFFFFFll) return fail(h, BJX_E_INVALID, "bad per_key");
  launch_prng_draw(2, keys, n_keys, per_key, out, pstream);
  BJX_CHECK_LAUNCH("k_prng_draw");
  return 0;
}

// ---- window adaptation ------------------------------------------------------------------------------------
extern "C" int bjx_da_init(bjx_handle_t h, float* st, const float* eps0, float* eps_out) {
  if (!h || !st || !eps0) return fail(h, BJX_E_INVALID, "null argument");
  BJX_CUDA(cudaSetDevice(h->cfg.device));
  launch_da(0, h->cfg.n_chains, st, eps0, 0.f, eps_out, h->stream);
  BJX_CHECK_LAUNCH("k_da_init");
  return 0;
}
extern "C" int bjx_da_update(bjx_handle_t h, float* st, const float* acc, float target, float* eps_out) {
  if (!h || !st || !acc) return fail(h, BJX_E_INVALID, "null argument");
  BJX_CUDA(cudaSetDevice(h->cfg.device));
  launch_da(1, h->cfg.n_chains, st, acc, target, eps_out, h->stream);
  BJX_CHECK_LAUNCH("k_da_update");
  return 0;
}
extern "C" int bjx_da_reset(bjx_handle_t h, float* st, float* eps_out) {
  if (!h || !st) return fail(h, BJX_E_INVALID, "null argument");
  BJX_CUDA(cudaSetDevice(h->cfg.device));
  launch_da(2, h->cfg.n_chains, st, nullptr, 0.f, eps_out, h->stream);
  BJX_CHECK_LAUNCH("k_da_reset");
  return 0;
}
extern "C" int bjx_da_final(bjx_handle_t h, const float* st, float* eps_out) {
  if (!h || !st || !eps_out) return fail(h, BJX_E_INVALID, "null argument");
  BJX_CUDA(cudaSetDevice(h->cfg.device));
  launch_da(3, h->cfg.n_chains, const_cast<float*>(st), nullptr, 0.f, eps_out, h->stream);
  BJX_CHECK_LAUNCH("k_da_final");
  return 0;
}
extern "C" int bjx_welford_update(bjx_handle_t h, const float* q, float* mean, float* m2, int32_t new_count) {
  if (!h || !q || !mean || !m2 || new_count < 1) return fail(h, BJX_E_INVALID, "bad argument");
  BJX_CUDA(cudaSetDevice(h->cfg.device));
  launch_welford_update((long long)h->cfg.n_chains * h->cfg.dim, q, mean, m2, new_count, h->stream);
  BJX_CHECK_LAUNCH("k_welford_update");
  return 0;
}
extern "C" int bjx_welford_final(bjx_handle_t h, float* mean, float* m2, int32_t count, float* imm_out) {
  if (!h || !mean || !m2 || !imm_out || count < 2) return fail(h, BJX_E_INVALID, "bad argument");
  BJX_CUDA(cudaSetDevice(h->cfg.device));
  launch_welford_final((long long)h->cfg.n_chains * h->cfg.dim, mean, m2, count, imm_out, h->stream);
  BJX_CHECK_LAUNCH("k_welford_final");
  return 0;
}
extern "C" int bjx_welford_dense_update(bjx_handle_t h, const float* q, float* mean, float* m2, int32_t new_count) {
  if (!h || !q || !mean || !m2 || new_count < 1) return fail(h, BJX_E_INVALID, "bad argument");
  BJX_CUDA(cudaSetDevice(h->cfg.device));
  launch_welford_dense_update(h->cfg.n_chains, h->cfg.dim, q, mean, m2, new_count, h->stream);
  BJX_CHECK_LAUNCH("k_welford_dense_m2");
  return 0;
}
extern "C" int bjx_welford_dense_final(bjx_handle_t h, float* mean, float* m2, int32_t count, float* imm_out) {
  if (!h || !mean || !m2 || !imm_out || count < 2) return fail(h, BJX_E_INVALID, "bad argument");
  BJX_CUDA(cudaSetDevice(h->cfg.device));
  launch_welford_dense_final(h->cfg.n_chains, h->cfg.dim, mean, m2, count, imm_out, h->stream);
  BJX_CHECK_LAUNCH("k_welford_dense_final");
  return 0;
}
extern "C" int bjx_pooled_stats(bjx_handle_t h, const float* q, const float* acc, float* out) {
  if (!h || !q || !acc || !out) return fail(h, BJX_E_INVALID, "null argument");
  BJX_CUDA(cudaSetDevice(h->cfg.device));
  launch_pooled_stats(h->cfg.n_chains, h->cfg.dim, q, acc, out, h->stream);
  BJX_CHECK_LAUNCH("k_pooled_stats");
  return 0;
}

extern "C" int bjx_pooled_stats_dense(bjx_handle_t h, const float* q, const float* acc, float* out) {
  if (!h || !q || !acc || !out) return fail(h, BJX_E_INVALID, "null argument");
  BJX_CUDA(cudaSetDevice(h->cfg.device));
  const size_t need = pooled_dense_scratch_floats(h->cfg.dim) * sizeof(float);
  if (h->pool_scratch_bytes < need) {
    if (h->pool_scratch) BJX_CUDA(cudaFree(h->pool_scratch));
    h->pool_scratch = nullptr;
    BJX_CUDA(cudaMalloc((void**)&h->pool_scratch, need));
    h->pool_scratch_bytes = need;
  }
  launch_pooled_stats_dense(h->cfg.n_chains, h->cfg.dim, q, acc, out, h->pool_scratch, h->stream);
  BJX_CHECK_LAUNCH("k_pooled_stats_dense");
  return 0;
}

// blackjax.diagnostics.potential_scale_reduction (diagnostics.py:39-89) for a history [T, C, D] (chain axis 1, sample
// axis 0): rhat_out [D].  scratch: device buffer of at least 2*C*D + 4 + 4*D floats.
extern "C" int bjx_potential_scale_reduction(bjx_handle_t h, const float* history, int32_t num_samples, float* rhat_out,
                                             float* scratch) {
  if (!h || !history || !rhat_out || !scratch) return fail(h, BJX_E_INVALID, "null argument");
  if (num_samples < 2 || h->cfg.n_chains < 2)
    return fail(h, BJX_E_INVALID, "potential_scale_reduction as implemented only works for two or more chains (and draws)");
  BJX_CUDA(cudaSetDevice(h->cfg.device));
  launch_rhat(num_samples, h->cfg.n_chains, h->cfg.dim, history, rhat_out, scratch, h->stream);
  BJX_CHECK_LAUNCH("k_rhat");
  return 0;
}

// blackjax.diagnostics.effective_sample_size (diagnostics.py:159-305) for a history [T, C, D] (chain axis 1, sample axis
// 0): ess_out [D].  scratch: 8-byte aligned device buffer of at least bjx_ess_scratch_floats(T, C, D) floats.
extern "C" int64_t bjx_ess_scratch_floats(int32_t num_samples, int32_t n_chains, int32_t dim) {
  return (int64_t)ess_scratch_floats(num_samples, n_chains, dim);
}
extern "C" int bjx_effective_sample_size(bjx_handle_t h, const float* history, int32_t num_samples, float* ess_out,
                                         float* scratch) {
  if (!h || !history || !ess_out || !scratch) return fail(h, BJX_E_INVALID, "null argument");
  if (num_samples < 2) return fail(h, BJX_E_INVALID, "The input array must have at least 2 samples");
  if ((reinterpret_cast<uintptr_t>(scratch) & 7u) != 0) return fail(h, BJX_E_INVALID, "scratch must be 8-byte aligned");
  BJX_CUDA(cudaSetDevice(h->cfg.device));
  launch_ess(num_samples, h->cfg.n_chains, h->cfg.dim, history, ess_out, scratch, h->stream);
  BJX_CHECK_LAUNCH("k_ess");
  return 0;
}

/* b200mcmc.h -- C ABI of libb200mcmc.so, the B200 (sm_100a) sampling path behind the
 * korentomas/mlx-mcmc Python API.
 *
 * The reference has no FFI layer: its boundary is the Python call convention
 *   MCMC(log_prob).run(...)            mlx_mcmc/inference/mcmc.py:38-189
 *   hmc / nuts / metropolis_hastings   mlx_mcmc/kernels/{hmc.py:7, nuts.py:16, metropolis.py:6}
 * and everything below it (mx.grad, elementwise MLX primitives, mx.random) lives in MLX.
 * This header is what a maintainer would bind (ctypes -- see INTEGRATION.md) to replace
 * that part.  Each entry point cites the reference code it replaces.
 *
 * Conventions
 *   - every function returns 0 on success; nonzero => b2m_last_error() (thread local text).
 *   - nothing throws across the ABI; the library never owns caller memory.
 *   - all `float*`/`double*`/`int*` in the *_args structs are DEVICE pointers allocated by the
 *     caller (torch CUDA tensors); `stream` is a cudaStream_t passed as void*.
 *   - one handle <-> one device; handles are not thread safe.
 *   - chains are independent; chain c of this process has global id chain_offset + c and its
 *     random stream depends only on (seed, global id, iteration, slot) -- never on the grid,
 *     the lanes-per-chain choice or the number of GPUs.
 */
#ifndef B200MCMC_H
#define B200MCMC_H

#ifdef __CUDACC_RTC__
/* NVRTC (the per-model pointwise kernels, mlx_mcmc_b200/jit.py) has no libc headers: the fixed-width types by hand */
typedef signed char int8_t;
typedef unsigned char uint8_t;
typedef int int32_t;
typedef unsigned int uint32_t;
typedef long long int64_t;
typedef unsigned long long uint64_t;
typedef unsigned long long uintptr_t;
#else
#include <stdint.h>
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define B2M_ABI_VERSION 4
#define B2M_MAX_TREE_DEPTH 12

/* ---- model description (produced by the Python tracer from the user's log_prob) ---- */

/* distribution tags: the reference's six classes (mlx_mcmc/distributions/<name>.py), plus Bernoulli (ABI 4) */
enum {
  B2M_NORMAL = 0,      /* normal.py:49-56      p0=loc  p1=scale               */
  B2M_HALFNORMAL = 1,  /* halfnormal.py:55-63  p0=scale           mask x>=0   */
  B2M_EXPONENTIAL = 2, /* exponential.py:61-71 p0=rate            mask x>=0   */
  B2M_GAMMA = 3,       /* gamma.py:53-88       p0=rate(beta) k0=alpha k1=lgamma(alpha)  mask x>0 */
  B2M_BETA = 4,        /* beta.py:53-91        k0=a k1=b k2=logB(a,b)         mask 0<x<1 */
  B2M_CONSTANT = 5,    /* a term with no traced operand: value k0 (Categorical with concrete
                          probs/index, categorical.py:69-93, folds to this)   */
  B2M_BERNOULLI = 7    /* x=label p0=logit: x p0 - softplus(p0), mask x in {0, 1}; p1 unused.  Not 6: that value is
                          B2M_SAMPLE_CATEGORICAL of b2m_sample, and 6 stays an unknown term tag */
};

/* operand kinds: value[n] of one slot of a term, n = element index inside the term */
enum {
  B2M_OP_CONST = 0,    /* c                                                    */
  B2M_OP_PARAM = 1,    /* theta[a]                                             */
  B2M_OP_DATA = 2,     /* arrays[a][n]                                         */
  B2M_OP_PARAMVEC = 3, /* theta[a + n]            (elementwise over a vector parameter) */
  B2M_OP_LIN = 4,      /* c + sum_{e in [a, a+b)} lin[e].coef * (lin[e].array>=0 ? arrays[.][n] : 1)
                            * (lin[e].param>=0 ? theta[lin[e].param] : 1)      */
  B2M_OP_MATVEC = 5    /* c + sum_d arrays[a][n, d] * theta[b + d]   (X @ beta; arrays[a] is [N, cols]) */
};

typedef struct {
  int32_t kind;
  int32_t a;
  int32_t b;
  float c;
} b2m_operand;

typedef struct {
  int32_t param; /* -1: no parameter factor */
  int32_t array; /* -1: no data factor      */
  float coef;
} b2m_lin_entry;

typedef struct {
  int32_t dist;
  int32_t length; /* elements summed by this term (1 for a scalar term) */
  float weight;   /* the term contributes weight * sum_n log p(x_n | ...) */
  float k0, k1, k2;
  b2m_operand x, p0, p1;
} b2m_term;

typedef struct {
  const float *data; /* device, row-major */
  int64_t rows;
  int64_t cols; /* 1 for a vector */
} b2m_array;

typedef struct b2m_model b2m_model;

/* Constraint transforms (SURVEY.md 8f row 3; the reference has none -- README.md:165,220, PROGRESS.md:119 list them as
 * planned).  With transforms set, the samplers move in the UNCONSTRAINED coordinate u_d and the model sees
 * theta_d = T_d(u_d); the log-Jacobian is added to log p and chained into the gradient.
 *   B2M_TF_LOG    theta = exp(u)        (support x > 0: HalfNormal / Exponential / Gamma values)   log|J| = u
 *   B2M_TF_LOGIT  theta = 1/(1+exp(-u)) (support 0 < x < 1: Beta values)                          log|J| = log theta + log(1-theta)
 * `theta` / `step_size` state of the sampler calls is then unconstrained; `draws` are written constrained unless
 * draws_unconstrained is set. */
enum { B2M_TF_NONE = 0, B2M_TF_LOG = 1, B2M_TF_LOGIT = 2 };

/* arithmetic of the two GLM contractions / evaluation path of pointwise models (were environment variables in ABI 1) */
enum { B2M_GLM_AUTO = 0, B2M_GLM_SIMT = 1, B2M_GLM_TC = 2, B2M_GLM_TC16 = 3 };
enum { B2M_POINTWISE_AUTO = 0, B2M_POINTWISE_GENERAL = 1 };
/* evaluation form of the GLM likelihood (DESIGN.md 4.2).  STREAM: two contractions over X per evaluation (B X^T with
 * the residual epilogue, then R X).  GRAM: one [C, D] x [D, D] contraction against X^T X, precomputed in float64 when
 * the model is created -- the Normal likelihood on the tensor-core paths only.  AUTO picks GRAM for a Normal likelihood
 * on a tensor-core path with N >= 2 D and D <= 4096 (padded), else STREAM.  Observation sharding (b2m_model_set_comm)
 * switches an AUTO model to STREAM; forcing GRAM where it cannot run is an error. */
enum { B2M_FORM_AUTO = 0, B2M_FORM_STREAM = 1, B2M_FORM_GRAM = 2 };

typedef struct {
  int32_t glm_path;          /* B2M_GLM_*: AUTO = tcgen05 3xFP16 when the data's dynamic range allows, else 3xTF32 */
  int32_t pointwise_path;    /* B2M_POINTWISE_*: AUTO = compact (registers + constant bank) when the model allows */
  const int32_t *transforms; /* HOST array [D] of B2M_TF_*, or NULL (= the reference: no transforms) */
  int32_t glm_form;          /* B2M_FORM_*: evaluation form of a GLM-class model with a Normal likelihood, see below */
  int32_t reserved[3];       /* must be zero */
} b2m_model_options;

/* ---- sampler arguments ---- */

enum {
  B2M_ADAPT_NONE = 0,
  B2M_ADAPT_REFERENCE = 1,      /* HMC: the +-5 % rule of hmc.py:164-170, per chain */
  B2M_ADAPT_DUAL_AVERAGING = 2, /* per chain: every chain is an independent replica of the reference's recurrences */
  B2M_ADAPT_POOLED = 3          /* NUTS, GLM class: ONE dual-averaging state driven by the mean acceptance statistic
                                   over the chains of the call; all chains share the step size (keeps a lock-step
                                   batch at one tree depth).  An extension: the reference has a single chain. */
};
enum { B2M_COMPAT_REFERENCE = 0, B2M_COMPAT_CORRECT = 1 };
enum { B2M_SCHED_ASYNC = 0, B2M_SCHED_SYNC = 1 };
/* B2M_SLICE_PEER: gradients travel through the peer window (b2m_model_peer_attach): K6's epilogue stores each finished
 * tile into its owner's slot over NVLink, no collective on the critical path.  B2M_SLICE_NCCL: reduce-scatter + all-gather. */
enum { B2M_SLICE_OFF = 0, B2M_SLICE_NCCL = 1, B2M_SLICE_PEER = 2 };

/* Replaces hmc()'s warm-up and sampling loops, kernels/hmc.py:155-198, with hmc_step :113-153,
 * leapfrog_step :69-100, hamiltonian :102-111 and the +-5 % rule :164-170 inside one launch. */
typedef struct {
  int64_t n_chains;     /* chains in this call (local)                                       */
  int64_t chain_offset; /* global id of local chain 0                                        */
  int64_t iter_offset;  /* global iteration index of the first iteration of this call        */
  int32_t n_iter;       /* iterations to run                                                 */
  int32_t n_leapfrog;   /* L                                                                 */
  int32_t adapt;        /* B2M_ADAPT_*: applied during this call (warm-up) or not (sampling) */
  int32_t lanes;        /* lanes per chain: 0 = library picks, else 1,2,4,8,16,32            */
  double target_accept;
  uint64_t seed;
  float *theta;        /* [n_chains, D] in/out                                                */
  double *step_size;   /* [n_chains] in/out                                                   */
  int64_t *n_accept;   /* [n_chains] in/out (cumulative accepted, drives the +-5 % rule)      */
  int64_t *n_total;    /* [n_chains] in/out                                                   */
  double *da_state;    /* [n_chains, 3] (H_bar, log eps_bar, mu) for dual averaging, or NULL  */
  float *draws;        /* [n_iter, n_chains, D] or NULL (warm-up)                             */
  const float *inj_normal;  /* [n_iter, n_chains, D] momentum draws to use instead of Philox, or NULL */
  const float *inj_uniform; /* [n_iter, n_chains]    accept uniforms, or NULL                 */
  float *trace_energy;      /* [n_iter, n_chains, 2] (H_init, H_prop) or NULL                 */
  uint8_t *trace_accept;    /* [n_iter, n_chains] or NULL                                     */
  /* ABI 2 */
  const float *inv_mass;    /* [D] diagonal of M^-1 shared by all chains (p ~ N(0, M), K = p'M^-1 p / 2, dq = eps M^-1 p),
                               or NULL = identity (the reference, hmc.py:102-111) */
  int32_t draws_unconstrained; /* models with transforms: write u instead of theta into `draws` (warm-up windows) */
  int32_t _pad2;
  int64_t adapt_origin;     /* dual averaging counts iterations from this global iteration (restart after a mass-matrix
                               update); 0 = the reference's single run */
} b2m_hmc_args;

/* Replaces metropolis_hastings(), kernels/metropolis.py:6-101 (proposal :66-74, accept :77-88). */
typedef struct {
  int64_t n_chains;
  int64_t chain_offset;
  int64_t iter_offset;
  int32_t n_iter;
  int32_t lanes;
  float proposal_scale;
  int32_t _pad;
  uint64_t seed;
  float *theta;       /* [n_chains, D] in/out */
  float *logp;        /* [n_chains] in/out: cached current log-prob (metropolis.py:55); NaN => recompute */
  int64_t *n_accept;  /* [n_chains] in/out */
  float *draws;       /* [n_iter, n_chains, D] or NULL */
  const float *inj_normal;  /* [n_iter, n_chains, D] or NULL */
  const float *inj_uniform; /* [n_iter, n_chains] or NULL */
  uint8_t *trace_accept;    /* [n_iter, n_chains] or NULL */
} b2m_mh_args;

/* Replaces nuts()'s loops, kernels/nuts.py:287-343, with nuts_step :220-285, build_tree :137-218
 * (iterative, one leaf per lock-step), no_u_turn :119-135 and dual averaging :62-68,298-310. */
typedef struct {
  int64_t n_chains;
  int64_t chain_offset;
  int64_t iter_offset;
  int32_t n_iter;
  int32_t max_tree_depth; /* <= B2M_MAX_TREE_DEPTH */
  int32_t adapt;          /* B2M_ADAPT_NONE, B2M_ADAPT_DUAL_AVERAGING (the reference's recurrences) or B2M_ADAPT_POOLED */
  int32_t compat;         /* B2M_COMPAT_REFERENCE: float32 slice underflow + NaN => alpha 1 (nuts.py:236-237,173)
                             B2M_COMPAT_CORRECT:   log-space slice, NaN => divergent, alpha 0 */
  int32_t lanes;
  float step_size_jitter; /* 0 = off (the reference).  > 0: every chain and iteration integrates with eps (1 + jitter (2u - 1)),
                             u from the spare word of Philox slot 0; adaptation keeps tracking the un-jittered eps.  Breaks the
                             resonance of the position-based U-turn test when a power of two steps is close to a whole
                             number of oscillation periods (DESIGN.md 4.2). */
  double target_accept;
  uint64_t seed;
  float *theta;        /* [n_chains, D] in/out */
  double *step_size;   /* [n_chains] in/out: eps used by the next iteration */
  double *da_state;    /* [n_chains, 3]: (H_bar, eps_bar, mu as float) in/out */
  int64_t *n_accept;   /* [n_chains] in/out: iterations with mean alpha > 0.5 (nuts.py:341) */
  int64_t *n_leaves;   /* [n_chains] in/out: leapfrog steps actually taken */
  int64_t *n_diverge;  /* [n_chains] in/out */
  float *draws;        /* [n_iter, n_chains, D] or NULL */
  int32_t *depths;     /* [n_iter, n_chains] or NULL */
  float *alphas;       /* [n_iter, n_chains] mean alpha, or NULL */
  /* draw injection (parity check 2); all NULL => Philox */
  const float *inj_normal; /* [n_iter, n_chains, D] */
  const float *inj_slice;  /* [n_iter, n_chains] */
  const float *inj_dir;    /* [n_iter, n_chains, max_tree_depth] */
  const float *inj_take;   /* [n_iter, n_chains, max_tree_depth] */
  const float *inj_merge;  /* [n_iter, n_chains, max_tree_depth, 2^max_tree_depth - 1] post-order merge slots */
  int32_t *trace_doubling; /* [n_iter, n_chains, max_tree_depth, 6] (v, n_sub, s_sub, took, s, n) or NULL */
  float *trace_energy;     /* [n_iter, n_chains] H0 or NULL */
  /* ABI 2 (the first three were environment variables in ABI 1) */
  const float *inv_mass;   /* [D] diagonal of M^-1 shared by all chains, or NULL = identity (the reference, nuts.py:113-117) */
  int32_t schedule;        /* GLM class: B2M_SCHED_ASYNC (iteration-asynchronous lock-step) or B2M_SCHED_SYNC */
  int32_t slice_state;     /* observation-sharded GLM models, adapt == NONE: rank r advances chains [r C/G, (r+1) C/G) only;
                              per-chain outputs are written by the owner (callers merge them).  B2M_SLICE_* */
  int32_t draws_unconstrained;
  int32_t _pad2;
  int64_t adapt_origin;    /* dual averaging (per chain or pooled) counts iterations from this global iteration: the
                              recurrences of nuts.py:298-310 see m = iteration - adapt_origin.  0 = the reference */
} b2m_nuts_args;

/* ---- entry points ---- */
#ifndef __CUDACC_RTC__   /* (the NVRTC-compiled per-model kernels include this header for the structs above only) */

const char *b2m_last_error(void);
int b2m_abi_version(void);
/* sizeof of the structs above as compiled, so a binding can verify its mirror */
int b2m_struct_sizes(int32_t *out6); /* term, operand, lin_entry, hmc_args, mh_args, nuts_args */
int b2m_options_size(void);          /* sizeof(b2m_model_options) */

/* Build a model from the traced term table.  Replaces the user log_prob + Distribution.log_prob
 * bodies (distributions/<name>.py) as differentiated by grad_log_prob, kernels/hmc.py:53-67.
 * `arrays[i].data` must stay valid for the life of the model. */
int b2m_model_create(const b2m_term *terms, int32_t n_terms, const b2m_lin_entry *lin, int32_t n_lin,
                     const b2m_array *arrays, int32_t n_arrays, int32_t D, const b2m_model_options *opt /* or NULL */,
                     b2m_model **out);
void b2m_model_destroy(b2m_model *m);
/* Per-model specialised kernels, pointwise class.  `cubin` = the translation unit mlx_mcmc_b200/jit.py generates from the
 * traced model (this library's own device headers with the term table baked in as literals, so the interpreter of the
 * generic kernels folds away) compiled by NVRTC for sm_100a; exports b2m_jit_logp_grad / _hmc / _mh / _nuts with the
 * parameter lists of the generic kernels.  Afterwards b2m_logp_grad / b2m_hmc_run / b2m_mh_run / b2m_nuts_run of this model
 * launch those entry points (same grid, same Philox slots, same arithmetic in the same order: bit-identical results).
 * The reference re-traces the Python log_prob on every gradient (kernels/hmc.py:53-67) and names JIT compilation as its
 * intended speed-up (TECHNICAL_OVERVIEW.md:232-236). */
int b2m_model_attach_module(b2m_model *m, const void *cubin, int64_t bytes, int32_t dmax);
int b2m_model_has_module(const b2m_model *m);
int b2m_model_dim(const b2m_model *m);
/* 0 = pointwise class (persistent register-resident kernels), 1 = GLM class (X @ beta, GEMM kernels) */
int b2m_model_class(const b2m_model *m);
/* GLM class: arithmetic of the two contractions -- 0 fp32 FMA tiles, 1 tcgen05 3xTF32, 2 tcgen05 3xFP16 (operands scaled
 * by powers of two into fp16's range, chosen automatically unless the data's dynamic range is too wide); -1 otherwise.
 * b2m_model_options.glm_path forces one. */
int b2m_model_glm_path(const b2m_model *m);
/* GLM class: evaluation form in use -- 1 streaming, 2 Gram (B2M_FORM_*); -1 otherwise */
int b2m_model_glm_form(const b2m_model *m);

/* log p(theta_c) and d/dtheta for C chains.  Replaces mx.grad(log_prob_flat)(*params) plus the
 * separate value call in hamiltonian() (kernels/hmc.py:53-67,102-111).  grad may be NULL. */
int b2m_logp_grad(b2m_model *m, const float *theta, int64_t n_chains, float *logp, float *grad,
                  int32_t lanes, void *stream);

/* ---- pointwise log-likelihood statistics over posterior draws (WAIC; DESIGN.md 4.6) ----
 * For every observation n of the listed observation terms -- terms whose value operand involves no parameter (CONST,
 * DATA, or LIN without parameter entries) while p0 or p1 does; CONSTANT terms never -- and every draw s:
 *     ll[s, n] = w log p(x_n | params(theta_s))      (w = the term's weight; theta_s in model coordinates: no transforms,
 *                                                      no Jacobian)
 * out[n] = (lppd_n, mean_n, var_n): log((1/S) sum_s exp ll[s, n]), (1/S) sum_s ll[s, n], and the sample variance (ddof 1)
 * over the S = n_draws draws.  Observations are numbered in term order, by element within a term.
 *   draws      DEVICE [n_draws, D] (the samplers' [S, C, D] seen as rows)
 *   obs_terms  HOST [n_obs_terms] term indices into the table given to b2m_model_create, increasing
 *   out        DEVICE [n_obs, 3] float64; n_obs must be the sum of the listed terms' lengths
 * The [S, N] matrix is never stored: GLM-class models reduce it inside the B X^T contraction (a statistics epilogue),
 * other terms in a SIMT kernel; float64 running state, fixed order: repeated calls are bit-identical.  Refused for
 * observation-sharded models.  Moves the GLM reference point beta0 (every sampler / logp call recentres). */
int b2m_loglik_stats(b2m_model *m, const float *draws, int64_t n_draws, const int32_t *obs_terms, int32_t n_obs_terms,
                     double *out, int64_t n_obs, void *stream);

int b2m_hmc_run(b2m_model *m, const b2m_hmc_args *a, void *stream);
int b2m_mh_run(b2m_model *m, const b2m_mh_args *a, void *stream);
int b2m_nuts_run(b2m_model *m, const b2m_nuts_args *a, void *stream);

/* ---- observation sharding (no reference counterpart: the reference is single device) ----
 * Every rank builds the model on its own row shard of (X, y) and holds every chain.  After b2m_model_set_comm each
 * value+gradient of a GLM-class model sums the [C, D] gradient partial and the [C] sum of squared residuals over
 * the ranks (one NCCL all-reduce on the caller's stream), so all ranks compute bit-identical results.
 * NCCL is bound at run time; without it these calls return an error and everything else keeps working. */
typedef struct b2m_comm b2m_comm;
int b2m_comm_unique_id(uint8_t *out128);                       /* rank 0 creates the 128-byte id; caller broadcasts it */
int b2m_comm_init(const uint8_t *id128, int32_t n_ranks, int32_t rank, b2m_comm **out);   /* collective */
void b2m_comm_destroy(b2m_comm *c);
int b2m_model_set_comm(b2m_model *m, b2m_comm *c, void *stream); /* collective (sums the shard row counts); c may be NULL */
int b2m_comm_allreduce_f32(b2m_comm *c, float *buf, int64_t n, void *stream);   /* in place, sum */

/* ---- peer window: the fused gradient exchange of observation sharding (B2M_SLICE_PEER) ----
 * Every rank allocates one window of b2m_model_peer_bytes() bytes (b2m_peer_alloc: cudaMalloc + a 64-byte CUDA IPC
 * handle), the handles travel over torch.distributed, every rank maps its peers' windows (b2m_peer_open) and hands the
 * G device pointers -- its own included, indexed by rank -- to b2m_model_peer_attach.  From then on a NUTS call with
 * slice_state = B2M_SLICE_PEER exchanges, per gradient, through plain NVLink stores:
 *   owner  -> all : the packed fp16 hi/lo position rows of its chains + row scales  (state kernel)
 *   all -> owner  : the [256, D] gradient tiles of the owner's chains, straight from K6's epilogue, and the sum z^2
 * with per-source slots summed in rank order by the owner (deterministic) and release/acquire flags at system scope. */
int b2m_peer_alloc(int64_t bytes, void **ptr, uint8_t *handle64);
int b2m_peer_open(const uint8_t *handle64, void **ptr);
int b2m_peer_close(void *ptr);
int b2m_peer_free(void *ptr);
int b2m_model_peer_bytes(b2m_model *m, int64_t n_chains, int32_t n_ranks, int64_t *bytes);
int b2m_model_peer_attach(b2m_model *m, void *const *windows, int32_t n_ranks, int32_t rank, int64_t n_chains, int64_t bytes);

/* ---- diagonal mass matrix from warm-up draws (SURVEY.md 8f row 3; reference roadmap README.md:165,220) ----
 * draws [S, C, D] (unconstrained coordinates) -> inv_mass[d] = regularised pooled variance over all S x C draws of
 * coordinate d around their grand mean:  v (n / (n + 5)) + 1e-3 (5 / (n + 5)), n = S x C  (Stan's shrinkage).
 * Two kernels: per-(slice, d) float64 partial moments in fixed order, then a fixed-order fold: deterministic. */
int b2m_mass_from_draws(const float *draws, int64_t S, int64_t C, int64_t D, float *inv_mass, void *stream);

/* ---- order statistics on the device (MCMC.summary: np.median / np.percentile, inference/mcmc.py:221-224) ----
 * x[n] float32 (device, not modified), q[n_q] in [0, 1] (host) -> out[n_q] (host) with numpy's default linear
 * interpolation between the two neighbouring order statistics.  Three 11/11/10-bit radix-histogram passes over x select
 * every requested order statistic at once (all n_q ranks share each pass). */
int b2m_quantiles(const float *x, int64_t n, const double *q, int32_t n_q, double *out, void *stream);

/* ---- forward sampling on the device (SURVEY.md 8f row 4) ----
 * n draws from one library distribution into out[n] (device).  Replaces Distribution.sample (distributions/<name>.py; the
 * reference's Gamma / Beta fall back to numpy, gamma.py:107-117, beta.py:110-119).  dist = B2M_NORMAL (p0 loc, p1 scale),
 * B2M_HALFNORMAL (p0 scale), B2M_EXPONENTIAL (p0 rate), B2M_GAMMA (p0 alpha, p1 rate), B2M_BETA (p0 a, p1 b),
 * B2M_BERNOULLI (p0 = probability of 1; draws are 0 / 1 as floats) or B2M_SAMPLE_CATEGORICAL (cdf = device array of n_cat cumulative probabilities, last = 1; draws are indices as floats).
 * Output i depends only on (seed, i). */
#define B2M_SAMPLE_CATEGORICAL 6
int b2m_sample(int32_t dist, float p0, float p1, const float *cdf, int32_t n_cat, uint64_t seed, int64_t n, float *out,
               void *stream);

/* ---- diagnostics on the device (SURVEY.md 8f) ----
 * draws is [S, C, D] as written by the samplers.
 * b2m_diag_series: per (chain, parameter) series -> mean [C, D], variance (ddof 0) [C, D], effective sample size by
 *   the reference's estimator (ess_mode 0: examples/06_nuts_comparison.py:22-41, 1: examples/02_hmc_comparison.py:111-128)
 *   and by Geyer's initial positive sequence; the two ESS outputs may be NULL.
 * b2m_diag_params: per parameter -> out[d][5] = pooled mean, pooled std (np.mean / np.std of
 *   mlx_mcmc/inference/mcmc.py:219-220 over all chains), Gelman-Rubin R-hat, ESS summed over chains (both estimators). */
int b2m_diag_series(const float *draws, int64_t S, int64_t C, int64_t D, int32_t ess_mode, float *mean, float *var,
                    float *ess_ref, float *ess_geyer, void *stream);
int b2m_diag_params(const float *mean, const float *var, const float *ess_ref, const float *ess_geyer, int64_t S,
                    int64_t C, int64_t D, double *out, void *stream);

/* Instrumentation: CUDA-event timing of every GEMM launch of the GLM class, on the launching stream.
 * b2m_profile(1) resets and starts recording, b2m_profile(0) stops; b2m_profile_read synchronises the device and
 * returns {K5 total ms, K5 launches, K6 total ms, K6 launches}. */
int b2m_profile(int32_t enable);
int b2m_profile_read(double *out4);
/* the same plus the per-chain kernels of the fused NUTS loop: {total ms, launches} x {K5, K6, state kernel, peer wait kernel
 * (includes waiting for the slowest rank's rows), peer signal kernel} */
int b2m_profile_read_ex(double *out10);

/* number of kernel launches this library has issued since load (bench.py's gpu_launches) */
int64_t b2m_launch_count(void);

#endif /* !__CUDACC_RTC__ */

#ifdef __cplusplus
}
#endif
#endif /* B200MCMC_H */

// GLM-class models: log p(theta) = priors(theta) + w * sum_n L(y_n | eta_n = c + (X @ beta)_n) with beta a slice of theta
// and one of two likelihood kinds (GlmModel::lik):
//     kLikNormal  Normal(y_n | eta_n, sigma), sigma a constant or a scalar parameter
//     kLikLogit   Bernoulli(y_n | logits = eta_n), labels y_n in {0, 1}
//
// The gradient of the likelihood is two dense contractions shared by all chains of a lock-step batch:
//     M = B X^T     [C, D] x [D, N]   -> residual epilogue, per element
//                                        Normal: R = w (y - c - M) / sigma_c^2,  ss_c += (y - c - M)^2
//                                        logit:  R = w (y - sigmoid(c + M)),     ss_c += y eta - softplus(eta)
//     G = R X       [C, N] x [N, D]
// (K5 / K6 of SURVEY.md 2b).  Two implementations sit behind the same interface:
//   * fp32 SIMT tiles (glm_simt.cu)    -- any shape, the validation path
//   * TMA + tcgen05 3xTF32 (glm_tc.cu) -- B, X, R split into tf32 hi + lo parts, fp32 accumulation in TMEM
#pragma once
#include <cuda_fp16.h>

#include "model.cuh"

namespace b2m {

struct Comm;  // comm.cu
int comm_unique_id(uint8_t *out128);
int comm_init(const uint8_t *id128, int nranks, int rank, Comm **out);
void comm_destroy(Comm *c);
int comm_nranks(const Comm *c);
int comm_rank(const Comm *c);
int comm_allgather_inplace(Comm *c, void *buf, int64_t count, int elt_bytes, cudaStream_t st);
int comm_reducescatter_f32_inplace(Comm *c, float *buf, int64_t count, cudaStream_t st);
int comm_allreduce_f32(Comm *c, float *buf, int64_t n, cudaStream_t st);
int comm_allreduce_i64(Comm *c, int64_t *buf, int64_t n, cudaStream_t st);
int comm_allreduce_f32_max(Comm *c, float *buf, int64_t n, cudaStream_t st);

constexpr int kCenterSlices = 32;  // chain slices of the deterministic two-stage mean (glm.cu, centring)
constexpr int kLikNormal = 0, kLikLogit = 1;   // GlmModel::lik
constexpr int kFormStream = 1, kFormGram = 2;   // GlmModel::form (b2m_model_options.glm_form: 0 = auto, 1, 2)
constexpr int kGramMaxDp = 4096;                // auto picks the Gram form up to this padded width (f64 G: 128 MB)
constexpr int kMaxPeers = 8;       // ranks of one NVSwitch box

// The peer window of observation sharding with sliced state (include/b200mcmc.h, B2M_SLICE_PEER).  Every rank owns one
// window with this layout; `base[s]` is rank s's window as mapped into this process (CUDA IPC), base[rank] is local.
struct PeerWindow {
  int nranks = 0, rank = 0;
  int64_t C = 0, own = 0;          // chains of the call, chains per owner (C / nranks)
  int Dp = 0;
  char *base[kMaxPeers] = {};
  // byte offsets inside a window
  size_t off_g = 0;      // float  [nranks][own][Dp]  gradient partial of MY chains from each source rank (unscaled)
  size_t off_ss = 0;     // float  [nranks][own]      sum z^2 partial of my chains from each source rank
  size_t off_bh = 0, off_bl = 0;   // __half [C][Dp]  packed position rows of ALL chains (each owner writes its rows everywhere)
  size_t off_meta = 0;   // float4 [C]                (1/sigma^2, 1 / row scale of delta', ||delta||^2, spare) per row
  size_t off_bflag = 0;  // u64 [nranks]  "rank s has published the rows of its chains for sequence number n"
  size_t off_gflag = 0;  // u64 [nranks]  "rank s has stored its gradient / sum z^2 partials of sequence number n"
  size_t off_done = 0;   // i64 [nranks]  finished chains of rank s's slice
  size_t off_err = 0;    // int           a spin-wait timed out (the call then fails instead of hanging the GPU)
  size_t bytes = 0;
  uint64_t seq = 0;      // sequence number of the last exchange (identical on every rank: the calls are collective)
};
size_t peer_layout(PeerWindow &w, int64_t C, int nranks, int Dp);

struct GlmModel {
  // problem
  int N = 0, D = 0;        // observations, regression coefficients
  int Np = 0, Dp = 0;      // padded: Np % 256 == 0, Dp % 64 == 0 (zero padded)
  int Dtot = 0;            // full parameter count
  int beta_off = 0;        // beta = theta[beta_off : beta_off + D]
  int sigma_param = -1;    // index of sigma in theta, or -1 when constant (always -1 for kLikLogit)
  float sigma_const = 1.f, loc_const = 0.f, weight = 1.f;
  int lik = kLikNormal;    // likelihood kind
  // observed data in HBM (owned by the handle)
  float *X = nullptr, *XT = nullptr;                         // [Np, Dp], [Dp, Np] fp32
  float *Xh = nullptr, *Xl = nullptr, *XTh = nullptr, *XTl = nullptr;  // tf32 hi / lo splits
  float *y = nullptr;                                        // [Np] observations / labels (padding: 0)
  // fp16 hi/lo encoding (use_tc == 2): X' = X * col_scale[d] (power of two, column maximum just below 2^14) split
  // into two halves, hi = fp16(x'), lo = fp16(x' - hi); same for the transposed copy
  __half *X16h = nullptr, *X16l = nullptr, *XT16h = nullptr, *XT16l = nullptr;
  float *col_scale = nullptr, *inv_col_scale = nullptr;      // [Dp]
  float *colmax = nullptr;                                   // [Dp] column maxima of |X| the scales were derived from
  float x_rownorm_max = 0.f;                                 // max_n ||X_n||_2: Cauchy-Schwarz bound of |(X delta)_n|
  unsigned *y0max_bits = nullptr;                            // device scalar: max_n |y0_n| as float bits (per recentre, Normal)
  // centring (glm.cu): beta0 = mean current position of the batch, float64 accumulation of
  //   Normal: y0 = y - c - X beta0        logit: y0 = eta0 = c + X beta0 (padding columns: -inf, which makes their
  //   log-likelihood and residual exactly zero in the epilogues without a per-element test)
  float *y0 = nullptr, *beta0 = nullptr;                     // [Np], [Dp]
  double *center_part = nullptr;                             // [32, Dp]
  // evaluation form (DESIGN.md 4.2).  Streaming: K5 (B X^T + residual epilogue) then K6 (R X), X read twice per leaf.
  // Gram (Normal likelihood, tensor-core paths, unsharded): with G = X^T X, b = X^T y0, q = ||y0||^2 precomputed,
  //     X^T (y0 - X delta) = b - G delta,   ||y0 - X delta||^2 = q - 2 delta.b + delta.(G delta)
  // so one [C, Dp] x [Dp, Dp] contraction per leaf replaces both passes over X.
  int form = kFormStream;
  int form_req = 0;                                          // the option as given (0 auto, 1 streaming, 2 Gram)
  double *G64 = nullptr;                                     // [Dp, Dp] X^T X, float64 sums of exact products
  double *gvec = nullptr;                                    // [2 Dp + 2] X^T y || X^T 1 || ||y||^2, sum y
  double *gb = nullptr;                                      // [Dp + 1] b = X^T y0 || q = ||y0||^2 (per recentre)
  double *gterm = nullptr;                                   // [Dp] per-coefficient terms of q (fixed-order sum)
  void *Gmh = nullptr, *Gml = nullptr;                       // [Dp, Dp] hi / lo halves of the B operand, row j = column j
                                                             // of diag(cs) G diag(cs) times t_j (fp16 or tf32 values)
  float *g_unscale = nullptr;                                // [Dp] 1 / (cs_j t_j)  (fp16 encoding; nullptr for tf32)
  // prior terms (everything except the matvec likelihood) as a pointwise term table
  KModel prior{};
  bool has_prior = false;
  // workspace sized for `cap` chains (padded to 128)
  int64_t cap = 0;
  float *B = nullptr, *Bh = nullptr, *Bl = nullptr;          // [cap, Dp]
  float *R = nullptr, *Rh = nullptr, *Rl = nullptr;          // [cap, Np]
  __half *B16h = nullptr, *B16l = nullptr;                   // [cap, Dp]  fp16 encoding of (beta - beta0) / col_scale * row scale
  __half *R16h = nullptr, *R16l = nullptr;                   // [cap, Np]  fp16 encoding of R * row scale
  float *a_unscale = nullptr, *r_scale = nullptr, *r_unscale = nullptr;   // [cap] per-row scales of the two A operands
  float *G = nullptr;                                        // [g_splits_cap, cap, Dp] split-K partials of the gradient
  int g_splits = 1, g_splits_cap = 1;
  float *ss_part = nullptr;                                  // [Np / 64, cap] per-column-tile partial sum of squares (Normal)
                                                             // or of the Bernoulli log-likelihood terms (logit)
  float *inv_var = nullptr;                                  // [cap]
  int use_tc = 0;                                            // 0: SIMT fp32 tiles, 1: tcgen05 3xTF32, 2: tcgen05 3xFP16
  // sampler workspace (glm_samplers.cu): one arena reused across calls, plus a pinned host flag
  char *ws = nullptr;
  size_t ws_cap = 0;
  int *h_flag = nullptr, *h_ring = nullptr;   // pinned: one flag + a ring of lagged counters
  const int *skip_flag = nullptr;             // device counter; the tensor-core contractions return at once when it has
  int skip_target = 0;                        // reached skip_target (set by the asynchronous NUTS loop only)
  // observation sharding (comm.cu): this handle holds rows [r0, r0 + N) of a model with N_total rows
  Comm *comm = nullptr;
  int64_t N_total = 0;
  float *red = nullptr;                                      // [cap * Dp + cap] gradient partial || sum z^2, all-reduced
  PeerWindow pw;                                             // attached by b2m_model_peer_attach (nranks == 0: none)
  // constraint transforms (include/b200mcmc.h): per-parameter B2M_TF_* codes, device [Dtot], or nullptr; the samplers'
  // theta is then the unconstrained coordinate and `thc` [cap, Dtot] holds T(theta) of the batch being evaluated
  int *tf = nullptr;
  float *thc = nullptr;
  // K6 push epilogue (peer window): set only while a peer-sliced NUTS call is running
  bool push_on = false;
  unsigned *blk_counter = nullptr;                           // device: "last block" counters of the signalling kernels
  volatile long long *h_prog = nullptr;                      // pinned + mapped: {ticks completed, finished chains} written by the device
};

int glm_set_comm(GlmModel &g, Comm *c, cudaStream_t st);
int glm_use_streaming(GlmModel &g, const char *why);   // observation sharding: back to the streaming form (or refuse)

int glm_reserve(GlmModel &g, int64_t n_chains);
void glm_free(GlmModel &g);

// log p and gradient for `theta` [C, Dtot] (device).  grad may be NULL.  recenter: move the reference point of
// the contraction to the mean of `theta` first (the samplers do it once per iteration, from the current states).
// idx / n_rows: evaluate only the chains idx[0..n_rows) (a compacted lock-step batch); outputs land at the chains' rows.
// own_count > 0 (observation sharding with sliced state, full batch only): the partial gradients are reduce-scattered
// and only the rows [own_base, own_base + own_count) -- this rank's chains -- are finished.
int glm_logp_grad(GlmModel &g, const float *theta, int64_t C, float *logp, float *grad, cudaStream_t st,
                  bool recenter = false, const int *idx = nullptr, int64_t n_rows = 0, int64_t own_base = 0,
                  int64_t own_count = 0);
int glm_recenter(GlmModel &g, const float *theta, int64_t C, cudaStream_t st);

// the two contractions (SIMT implementation)
int simt_gemm_resid(GlmModel &g, int64_t Cp, cudaStream_t st);   // B -> R, ss_part
int simt_gemm_grad(GlmModel &g, int64_t Cp, cudaStream_t st);    // R -> G
// tcgen05 implementation (glm_tc.cu)
int tc_gemm_resid(GlmModel &g, int64_t Cp, cudaStream_t st);     // B -> R, ss_part
int tc_gemm_grad(GlmModel &g, int64_t Cp, cudaStream_t st);      // R -> G
int tc_gemm_gram(GlmModel &g, int64_t Cp, cudaStream_t st);      // B -> G = (beta - beta0) G~  (Gram form)
// pointwise log-likelihood statistics over posterior draws (b2m_loglik_stats): B -> partials [Cp / 32, Np] of 32 draws
int simt_gemm_stats(GlmModel &g, int64_t Cp, int64_t rows_valid, float4 *part, cudaStream_t st);
int tc_gemm_stats(GlmModel &g, int64_t Cp, int64_t rows_valid, float4 *part, cudaStream_t st);
int glm_loglik_center(GlmModel &g, const float *draws, int64_t S, cudaStream_t st);   // beta0 = mean draw, y0 / eta0
int glm_loglik_batch(GlmModel &g, const float *draws, int64_t rows, float4 *part, cudaStream_t st);
bool tc_available();
void tc_profile(bool enable);
int tc_profile_read(double *out4);
int tc_profile_read_n(double *out, int n_kinds);
void prof_mark(int kind, cudaStream_t st);   // kinds 2 state, 3 peer wait, 4 peer signal: call before and after the launch
int grad_splits(const GlmModel &g, int64_t Cp, int k_blocks);
int contraction_splits(const GlmModel &g, int64_t Cp);   // split-K of the gradient contraction of the model's form

int tc_gemm_grad_push(GlmModel &g, int64_t Cp, cudaStream_t st);   // K6 whose epilogue stores into the owners' windows
int glm_finish_launch(GlmModel &g, const float *theta, int64_t C, float *logp, float *grad, cudaStream_t st,
                      const int *idx, int64_t n_rows);
int glm_hmc_run(GlmModel &g, const b2m_hmc_args &a, cudaStream_t st);
int glm_nuts_run(GlmModel &g, const b2m_nuts_args &a, cudaStream_t st);
int glm_mh_run(GlmModel &g, const b2m_mh_args &a, cudaStream_t st);

// round-to-nearest split of an fp32 value into two tf32-representable parts, x ~= hi + lo
__host__ __device__ inline void split_tf32(float x, float &hi, float &lo) {
  union { float f; uint32_t u; } a, b;
  a.f = x;
  a.u = (a.u + 0x00001000u) & 0xffffe000u;
  hi = a.f;
  b.f = x - hi;
  b.u = (b.u + 0x00001000u) & 0xffffe000u;
  lo = b.f;
}

}  // namespace b2m

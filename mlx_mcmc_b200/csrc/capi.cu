// C ABI of libb200mcmc.so (declared in include/b200mcmc.h): model handle, validation, dispatch.
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <string>
#include <vector>

#include "glm.cuh"

namespace b2m {

static thread_local std::string tl_error;
std::atomic<int64_t> g_launches{0};
void set_error(const std::string &msg) { tl_error = msg; }

int pick_lanes(const KModel &km, int64_t n_chains, int requested);
struct JitModule;
int jit_load(const void *image, int dmax, JitModule **out);
void jit_unload(JitModule *m);
int launch_logp_grad(const KModel &km, const float *theta, int64_t C, float *logp, float *grad, int lanes,
                     cudaStream_t st, JitModule *jit);
int launch_hmc(const KModel &km, b2m_hmc_args a, cudaStream_t st, JitModule *jit);
int launch_mh(const KModel &km, b2m_mh_args a, cudaStream_t st, JitModule *jit);
int launch_nuts(const KModel &km, b2m_nuts_args a, cudaStream_t st, JitModule *jit);
int glm_build(GlmModel &g, const float *X, const float *y, int N, int D, bool force_tc16);
int glm_check_labels(const float *y, int N);
int mass_from_draws(const float *draws, int64_t S, int64_t C, int64_t D, float *inv_mass, cudaStream_t st);
int quantiles(const float *x, int64_t n, const double *q, int n_q, double *out, cudaStream_t st);
int peer_alloc(int64_t bytes, void **ptr, uint8_t *handle64);
int peer_open(const uint8_t *handle64, void **ptr);
int peer_close(void *ptr);
int peer_free(void *ptr);
int glm_peer_attach(GlmModel &g, void *const *windows, int n_ranks, int rank, int64_t n_chains, int64_t bytes);
int debug_tc_gemm(const float *A, const float *Bm, int M, int N, int K, float *Cout, int chunk_kb, int mma_mask,
                  cudaStream_t st);

int sample(int dist, float p0, float p1, const float *cdf, int n_cat, uint64_t seed, int64_t n, float *out, cudaStream_t st);
int diag_series(const float *draws, int64_t S, int64_t C, int64_t D, int ess_mode, float *mean, float *var, float *ess_ref,
                float *ess_geyer, cudaStream_t st);
int diag_params(const float *mean, const float *var, const float *ess_ref, const float *ess_geyer, int64_t S, int64_t C,
                int64_t D, double *out, cudaStream_t st);
int loglik_stats(const KModel &km, GlmModel *g, int lik, const std::vector<b2m_term> &terms, const std::vector<int> &obs,
                 const float *draws, int64_t S, double *out, int64_t n_obs, cudaStream_t st);

}  // namespace b2m

struct b2m_model {
  b2m::KModel km{};
  int model_class = 0;
  void *dev_terms = nullptr, *dev_lin = nullptr, *dev_arrays = nullptr;
  std::vector<b2m_term> terms;
  std::vector<b2m_lin_entry> lin;
  std::vector<b2m_array> arrays;
  b2m::GlmModel glm;           // model_class == 1
  void *dev_prior_terms = nullptr;
  b2m::JitModule *jit = nullptr;   // per-model specialised kernels (b2m_model_attach_module), pointwise class
  // A handle is NOT re-entrant: GLM-class models keep one workspace arena, one progress ring and one peer window per
  // handle.  Entry points that use them take this lock without waiting; a second concurrent call on the same handle is an
  // error (use one handle per thread / stream), never silent corruption.
  std::mutex busy;
};

#define B2M_MODEL_GUARD(m)                                                                               \
  std::unique_lock<std::mutex> _guard((m)->busy, std::try_to_lock);                                      \
  B2M_REQUIRE(_guard.owns_lock(), "this model handle is in use by another call (handles are not re-entrant: one per thread)")

using b2m::set_error;

// Observation terms (b2m_loglik_stats; the Python tracer's TracedModel.observation_terms makes the same choice): the
// value operand involves no parameter and at least one of the distribution's parameters does.  Constant terms never.
static bool op_has_param(const b2m_operand &o, const std::vector<b2m_lin_entry> &lin) {
  if (o.kind == B2M_OP_PARAM || o.kind == B2M_OP_PARAMVEC || o.kind == B2M_OP_MATVEC) return true;
  if (o.kind == B2M_OP_LIN)
    for (int e = o.a; e < o.a + o.b; ++e)
      if (lin[e].param >= 0) return true;
  return false;
}
static bool is_observation_term(const b2m_term &T, const std::vector<b2m_lin_entry> &lin) {
  return T.dist != B2M_CONSTANT && !op_has_param(T.x, lin) && (op_has_param(T.p0, lin) || op_has_param(T.p1, lin));
}

static bool valid_lanes(int l) { return l == 0 || l == 1 || l == 2 || l == 4 || l == 8 || l == 16 || l == 32; }

static int check_operand(const b2m_operand &o, int length, int D, int n_lin, const b2m_array *arrays, int n_arrays,
                         const char *slot, int t) {
  auto fail = [&](const std::string &why) {
    set_error("term " + std::to_string(t) + " operand " + slot + ": " + why);
    return 1;
  };
  switch (o.kind) {
    case B2M_OP_CONST: return 0;
    case B2M_OP_PARAM:
      if (o.a < 0 || o.a >= D) return fail("parameter index out of range");
      return 0;
    case B2M_OP_DATA:
      if (o.a < 0 || o.a >= n_arrays) return fail("array index out of range");
      if (arrays[o.a].cols != 1 || arrays[o.a].rows < length) return fail("observed array shorter than the term");
      return 0;
    case B2M_OP_PARAMVEC:
      if (o.a < 0 || o.a + length > D) return fail("parameter slice out of range");
      return 0;
    case B2M_OP_LIN:
      if (o.a < 0 || o.b < 0 || o.a + o.b > n_lin) return fail("linear-entry range out of range");
      return 0;
    case B2M_OP_MATVEC:
      if (o.a < 0 || o.a >= n_arrays) return fail("matrix index out of range");
      if (arrays[o.a].rows < length) return fail("matrix has fewer rows than the term");
      if (o.b < 0 || o.b + arrays[o.a].cols > D) return fail("matvec parameter slice out of range");
      return 0;
    default: return fail("unknown operand kind " + std::to_string(o.kind));
  }
}

// GLM class: exactly one likelihood over X @ beta (+ const) and an observed vector y -- a Normal with X @ beta as its
// location and a constant or scalar-parameter scale, or a Bernoulli with X @ beta as its logits and labels y in {0, 1};
// every other term is a pointwise prior.
static int setup_glm(b2m_model *m, int D, int glm_path, int glm_form, const int32_t *tf) {
  int lik = -1;
  for (size_t t = 0; t < m->terms.size(); ++t) {
    const b2m_term &T = m->terms[t];
    const bool has_mv = T.x.kind == B2M_OP_MATVEC || T.p0.kind == B2M_OP_MATVEC || T.p1.kind == B2M_OP_MATVEC;
    if (!has_mv) continue;
    B2M_REQUIRE(lik < 0, "GLM class: only one X @ beta term is supported");
    const bool normal = T.dist == B2M_NORMAL && (T.p1.kind == B2M_OP_CONST || T.p1.kind == B2M_OP_PARAM);
    B2M_REQUIRE((normal || T.dist == B2M_BERNOULLI) && T.p0.kind == B2M_OP_MATVEC && T.x.kind == B2M_OP_DATA,
                "GLM class: X @ beta must be the location of a Normal likelihood over an observed vector, with a "
                "constant or scalar-parameter scale, or the logits of a Bernoulli likelihood over observed labels");
    lik = (int)t;
  }
  B2M_REQUIRE(lik >= 0, "GLM class: no X @ beta term found");
  const b2m_term &L = m->terms[lik];
  const b2m_array &X = m->arrays[L.p0.a];
  const b2m_array &Y = m->arrays[L.x.a];
  B2M_REQUIRE(X.rows == L.length && Y.rows >= L.length, "GLM class: X rows / y length do not match the term length");
  b2m::GlmModel &g = m->glm;
  g.Dtot = D;
  g.beta_off = L.p0.b;
  g.loc_const = L.p0.c;
  g.weight = L.weight;
  g.lik = L.dist == B2M_BERNOULLI ? b2m::kLikLogit : b2m::kLikNormal;
  g.sigma_param = (g.lik == b2m::kLikNormal && L.p1.kind == B2M_OP_PARAM) ? L.p1.a : -1;
  g.sigma_const = (g.lik == b2m::kLikNormal && L.p1.kind == B2M_OP_CONST) ? L.p1.c : 1.f;
  if (g.lik == b2m::kLikLogit)
    if (int rc = b2m::glm_check_labels(Y.data, (int)L.length)) return rc;
  // b2m_model_options.glm_path: SIMT (fp32 FMA tiles) | TC (tcgen05 3xTF32) | TC16 (tcgen05 3xFP16 with scaled operands);
  // AUTO: the fp16 encoding when the data's dynamic range allows it (checked in glm_build), else tf32
  g.use_tc = (!b2m::tc_available() || glm_path == B2M_GLM_SIMT) ? 0 : (glm_path == B2M_GLM_TC ? 1 : 2);
  g.form_req = glm_form;   // resolved in glm_build once the encoding is known
  if (tf) {   // constraint transforms: device copy of the per-parameter codes (before any workspace is reserved)
    bool any = false;
    for (int d = 0; d < D; ++d) any = any || tf[d] != B2M_TF_NONE;
    if (any) {
      B2M_CHECK_CUDA(cudaMalloc(reinterpret_cast<void **>(&g.tf), sizeof(int) * D));
      B2M_CHECK_CUDA(cudaMemcpy(g.tf, tf, sizeof(int) * D, cudaMemcpyHostToDevice));
    }
  }
  if (int rc = b2m::glm_build(g, X.data, Y.data, (int)L.length, (int)X.cols, glm_path == B2M_GLM_TC16)) return rc;
  // prior = all other terms
  std::vector<b2m_term> prior;
  for (size_t t = 0; t < m->terms.size(); ++t)
    if ((int)t != lik) prior.push_back(m->terms[t]);
  g.has_prior = !prior.empty();
  g.prior = m->km;
  g.prior.n_terms = (int)prior.size();
  g.prior.max_len = 1;
  if (g.has_prior) {
    B2M_CHECK_CUDA(cudaMalloc(&m->dev_prior_terms, sizeof(b2m_term) * prior.size()));
    B2M_CHECK_CUDA(cudaMemcpy(m->dev_prior_terms, prior.data(), sizeof(b2m_term) * prior.size(), cudaMemcpyHostToDevice));
    g.prior.terms = static_cast<const b2m_term *>(m->dev_prior_terms);
    // 1-D arrays used by the priors are small; the big matrices are never staged (cols != 1) but y is 1-D:
    // disable staging when it would not fit
    int64_t stage = 0;
    for (auto &a : m->arrays) if (a.cols == 1) stage += (a.rows + 3) & ~int64_t(3);
    g.prior.stage_floats = (stage * 4 <= 32 * 1024) ? (int32_t)stage : 0;
  }
  return 0;
}

extern "C" {

const char *b2m_last_error(void) { return b2m::tl_error.c_str(); }
int b2m_abi_version(void) { return B2M_ABI_VERSION; }
int64_t b2m_launch_count(void) { return b2m::g_launches.load(); }

// Internal (not part of the public header): C[M,N] = A[M,K] . B[N,K]^T through the 3xTF32 tcgen05 kernel, with the
// promotion interval and the set of partial products selectable, for accuracy experiments and tests.
int b2m_debug_tc_gemm(const float *A, const float *Bm, int M, int N, int K, float *C, int chunk_kb, int mma_mask,
                      void *stream) {
  return b2m::debug_tc_gemm(A, Bm, M, N, K, C, chunk_kb, mma_mask, static_cast<cudaStream_t>(stream));
}

int b2m_sample(int32_t dist, float p0, float p1, const float *cdf, int32_t n_cat, uint64_t seed, int64_t n, float *out,
               void *stream) {
  B2M_REQUIRE(n >= 0 && (out || n == 0), "b2m_sample: bad output");
  B2M_REQUIRE((dist >= B2M_NORMAL && dist <= B2M_BETA) || dist == B2M_SAMPLE_CATEGORICAL || dist == B2M_BERNOULLI,
              "b2m_sample: unknown distribution tag");
  if (dist == B2M_BERNOULLI) B2M_REQUIRE(p0 >= 0.f && p0 <= 1.f, "b2m_sample: a Bernoulli probability must lie in [0, 1]");
  B2M_REQUIRE(dist != B2M_SAMPLE_CATEGORICAL || (cdf && n_cat > 0), "b2m_sample: categorical needs a cdf");
  if (dist == B2M_GAMMA || dist == B2M_BETA) B2M_REQUIRE(p0 > 0.f && p1 > 0.f, "b2m_sample: shape / rate parameters must be positive");
  return b2m::sample(dist, p0, p1, cdf, n_cat, seed, n, out, static_cast<cudaStream_t>(stream));
}

int b2m_diag_series(const float *draws, int64_t S, int64_t C, int64_t D, int32_t ess_mode, float *mean, float *var,
                    float *ess_ref, float *ess_geyer, void *stream) {
  B2M_REQUIRE(draws && mean && var, "b2m_diag_series: NULL argument");
  B2M_REQUIRE(S > 0 && C > 0 && D > 0, "b2m_diag_series: sizes must be positive");
  B2M_REQUIRE(ess_mode == 0 || ess_mode == 1, "b2m_diag_series: ess_mode must be 0 or 1");
  return b2m::diag_series(draws, S, C, D, ess_mode, mean, var, ess_ref, ess_geyer, static_cast<cudaStream_t>(stream));
}

int b2m_diag_params(const float *mean, const float *var, const float *ess_ref, const float *ess_geyer, int64_t S,
                    int64_t C, int64_t D, double *out, void *stream) {
  B2M_REQUIRE(mean && var && out, "b2m_diag_params: NULL argument");
  B2M_REQUIRE(S > 0 && C > 0 && D > 0, "b2m_diag_params: sizes must be positive");
  return b2m::diag_params(mean, var, ess_ref, ess_geyer, S, C, D, out, static_cast<cudaStream_t>(stream));
}

int b2m_profile(int32_t enable) {
  b2m::tc_profile(enable != 0);
  return 0;
}

int b2m_profile_read(double *out4) {
  B2M_REQUIRE(out4 != nullptr, "b2m_profile_read: NULL argument");
  return b2m::tc_profile_read(out4);
}

int b2m_profile_read_ex(double *out10) {
  B2M_REQUIRE(out10 != nullptr, "b2m_profile_read_ex: NULL argument");
  return b2m::tc_profile_read_n(out10, 5);
}

int b2m_struct_sizes(int32_t *out6) {
  out6[0] = (int32_t)sizeof(b2m_term);
  out6[1] = (int32_t)sizeof(b2m_operand);
  out6[2] = (int32_t)sizeof(b2m_lin_entry);
  out6[3] = (int32_t)sizeof(b2m_hmc_args);
  out6[4] = (int32_t)sizeof(b2m_mh_args);
  out6[5] = (int32_t)sizeof(b2m_nuts_args);
  return 0;
}

int b2m_options_size(void) { return (int)sizeof(b2m_model_options); }

int b2m_model_create(const b2m_term *terms, int32_t n_terms, const b2m_lin_entry *lin, int32_t n_lin,
                     const b2m_array *arrays, int32_t n_arrays, int32_t D, const b2m_model_options *opt, b2m_model **out) {
  B2M_REQUIRE(out != nullptr, "b2m_model_create: out is NULL");
  *out = nullptr;
  b2m_model_options o{};
  if (opt) o = *opt;
  B2M_REQUIRE(o.glm_path >= B2M_GLM_AUTO && o.glm_path <= B2M_GLM_TC16, "b2m_model_create: unknown glm_path");
  B2M_REQUIRE(o.pointwise_path == B2M_POINTWISE_AUTO || o.pointwise_path == B2M_POINTWISE_GENERAL,
              "b2m_model_create: unknown pointwise_path");
  B2M_REQUIRE(o.glm_form >= B2M_FORM_AUTO && o.glm_form <= B2M_FORM_GRAM, "b2m_model_create: unknown glm_form");
  for (int i = 0; i < 3; ++i) B2M_REQUIRE(o.reserved[i] == 0, "b2m_model_create: reserved option fields must be zero");
  if (o.transforms)
    for (int d = 0; d < D; ++d)
      B2M_REQUIRE(o.transforms[d] >= B2M_TF_NONE && o.transforms[d] <= B2M_TF_LOGIT, "b2m_model_create: unknown transform code");
  B2M_REQUIRE(n_terms > 0 && n_terms <= 256, "b2m_model_create: need 1..256 terms");
  B2M_REQUIRE(D > 0, "b2m_model_create: D must be positive");
  B2M_REQUIRE(n_lin >= 0 && n_arrays >= 0, "b2m_model_create: negative table size");
  int n_matvec = 0, max_len = 1;
  for (int e = 0; e < n_lin; ++e) {
    B2M_REQUIRE(lin[e].param < D, "linear entry: parameter index out of range");
    B2M_REQUIRE(lin[e].array < n_arrays, "linear entry: array index out of range");
  }
  for (int t = 0; t < n_terms; ++t) {
    const b2m_term &T = terms[t];
    if ((T.dist < B2M_NORMAL || T.dist > B2M_CONSTANT) && T.dist != B2M_BERNOULLI) {
      set_error("term " + std::to_string(t) + ": unknown distribution tag " + std::to_string(T.dist));
      return 1;
    }
    B2M_REQUIRE(T.length >= 0, "term length must be non-negative");
    if (check_operand(T.x, T.length, D, n_lin, arrays, n_arrays, "x", t)) return 1;
    if (check_operand(T.p0, T.length, D, n_lin, arrays, n_arrays, "p0", t)) return 1;
    if (check_operand(T.p1, T.length, D, n_lin, arrays, n_arrays, "p1", t)) return 1;
    n_matvec += (T.x.kind == B2M_OP_MATVEC) + (T.p0.kind == B2M_OP_MATVEC) + (T.p1.kind == B2M_OP_MATVEC);
    if (T.length > max_len) max_len = T.length;
  }
  b2m_model *m = new b2m_model();
  m->terms.assign(terms, terms + n_terms);
  if (n_lin) m->lin.assign(lin, lin + n_lin);
  if (n_arrays) m->arrays.assign(arrays, arrays + n_arrays);
  m->model_class = n_matvec > 0 ? 1 : 0;

  std::vector<b2m::DevArray> da(n_arrays > 0 ? n_arrays : 1);
  int64_t stage = 0;
  for (int a = 0; a < n_arrays; ++a) {
    da[a].ptr = arrays[a].data;
    da[a].rows = arrays[a].rows;
    da[a].cols = arrays[a].cols;
    if (arrays[a].cols == 1) stage += (arrays[a].rows + 3) & ~int64_t(3);
  }
  auto up = [&](void **dst, const void *src, size_t bytes) -> int {
    if (bytes == 0) bytes = 16;
    B2M_CHECK_CUDA(cudaMalloc(dst, bytes));
    if (src) B2M_CHECK_CUDA(cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice));
    return 0;
  };
  if (up(&m->dev_terms, terms, sizeof(b2m_term) * n_terms) ||
      up(&m->dev_lin, n_lin ? lin : nullptr, sizeof(b2m_lin_entry) * n_lin) ||
      up(&m->dev_arrays, n_arrays ? da.data() : nullptr, sizeof(b2m::DevArray) * n_arrays)) {
    b2m_model_destroy(m);
    return 2;
  }
  m->km.terms = static_cast<const b2m_term *>(m->dev_terms);
  m->km.lin = static_cast<const b2m_lin_entry *>(m->dev_lin);
  m->km.arrays = static_cast<const b2m::DevArray *>(m->dev_arrays);
  m->km.n_terms = n_terms;
  m->km.n_lin = n_lin;
  m->km.n_arrays = n_arrays;
  m->km.D = D;
  m->km.max_len = max_len;
  // compact models: the table rides in the kernel parameters (model.cuh)
  bool compact = n_terms <= b2m::kCompactTerms && D <= b2m::kCompactDim && n_matvec == 0;
  for (int t = 0; t < n_terms && compact; ++t)
    compact = terms[t].x.kind != B2M_OP_LIN && terms[t].p0.kind != B2M_OP_LIN && terms[t].p1.kind != B2M_OP_LIN;
  if (o.pointwise_path == B2M_POINTWISE_GENERAL) compact = false;
  m->km.compact = compact ? 1 : 0;
  m->km.has_tf = 0;
  memset(m->km.tf, 0, sizeof(m->km.tf));
  if (o.transforms && n_matvec == 0) {
    for (int d = 0; d < D; ++d)
      if (o.transforms[d] != B2M_TF_NONE) {
        if (d >= 16) {
          set_error("constraint transforms: pointwise models support at most 16 scalar parameters");
          b2m_model_destroy(m);
          return 1;
        }
        m->km.tf[d] = (uint8_t)o.transforms[d];
        m->km.has_tf = 1;
      }
  }
  memset(m->km.cterms, 0, sizeof(m->km.cterms));
  if (compact) memcpy(m->km.cterms, terms, sizeof(b2m_term) * n_terms);
  // observation vectors are staged in shared memory when they fit beside the mailboxes
  m->km.stage_floats = (stage * 4 <= 96 * 1024) ? (int32_t)stage : 0;
  if (m->model_class == 1) {
    if (int rc = setup_glm(m, D, o.glm_path, o.glm_form, o.transforms)) {
      b2m_model_destroy(m);
      return rc;
    }
  }
  *out = m;
  return 0;
}

void b2m_model_destroy(b2m_model *m) {
  if (!m) return;
  if (m->dev_terms) cudaFree(m->dev_terms);
  if (m->dev_lin) cudaFree(m->dev_lin);
  if (m->dev_arrays) cudaFree(m->dev_arrays);
  if (m->dev_prior_terms) cudaFree(m->dev_prior_terms);
  if (m->model_class == 1) b2m::glm_free(m->glm);
  b2m::jit_unload(m->jit);
  delete m;
}

int b2m_model_attach_module(b2m_model *m, const void *cubin, int64_t bytes, int32_t dmax) {
  B2M_REQUIRE(m && cubin && bytes > 0, "b2m_model_attach_module: bad argument");
  B2M_REQUIRE(m->model_class == 0, "b2m_model_attach_module: specialised kernels exist for the pointwise class only");
  B2M_REQUIRE(dmax == 2 || dmax == 4 || dmax == 8 || dmax == 16, "b2m_model_attach_module: dmax must be 2, 4, 8 or 16");
  B2M_REQUIRE(dmax >= m->km.D, "b2m_model_attach_module: dmax is smaller than the model's parameter count");
  b2m::JitModule *j = nullptr;
  if (int rc = b2m::jit_load(cubin, dmax, &j)) return rc;
  b2m::jit_unload(m->jit);
  m->jit = j;
  return 0;
}
int b2m_model_has_module(const b2m_model *m) { return (m && m->jit) ? 1 : 0; }

int b2m_model_dim(const b2m_model *m) { return m ? m->km.D : -1; }
int b2m_model_class(const b2m_model *m) { return m ? m->model_class : -1; }
int b2m_model_glm_path(const b2m_model *m) { return (m && m->model_class == 1) ? m->glm.use_tc : -1; }
int b2m_model_glm_form(const b2m_model *m) { return (m && m->model_class == 1) ? m->glm.form : -1; }

int b2m_logp_grad(b2m_model *m, const float *theta, int64_t n_chains, float *logp, float *grad, int32_t lanes,
                  void *stream) {
  B2M_REQUIRE(m && theta && logp, "b2m_logp_grad: NULL argument");
  B2M_REQUIRE(n_chains > 0, "b2m_logp_grad: n_chains must be positive");
  B2M_REQUIRE(valid_lanes(lanes), "b2m_logp_grad: lanes must be 0 or a power of two <= 32");
  B2M_MODEL_GUARD(m);
  if (m->model_class == 1)
    return b2m::glm_logp_grad(m->glm, theta, n_chains, logp, grad, static_cast<cudaStream_t>(stream), true);
  return b2m::launch_logp_grad(m->km, theta, n_chains, logp, grad, lanes, static_cast<cudaStream_t>(stream), m->jit);
}

int b2m_loglik_stats(b2m_model *m, const float *draws, int64_t n_draws, const int32_t *obs_terms, int32_t n_obs_terms,
                     double *out, int64_t n_obs, void *stream) {
  B2M_REQUIRE(m && draws && obs_terms && out, "b2m_loglik_stats: NULL argument");
  B2M_REQUIRE(n_draws > 0, "b2m_loglik_stats: n_draws must be positive");
  B2M_REQUIRE(n_obs_terms > 0, "b2m_loglik_stats: no observation terms listed");
  B2M_REQUIRE(m->model_class == 0 || (m->glm.comm == nullptr && m->glm.pw.nranks == 0),
              "b2m_loglik_stats: the model is observation-sharded (each rank holds only its rows of the observations)");
  const int n_terms = (int)m->terms.size();
  std::vector<int> obs(n_obs_terms);
  int64_t total = 0;
  for (int i = 0; i < n_obs_terms; ++i) {
    const int t = obs_terms[i];
    if (t < 0 || t >= n_terms) {
      set_error("b2m_loglik_stats: term index " + std::to_string(t) + " out of range (the model has " +
                std::to_string(n_terms) + " terms)");
      return 1;
    }
    if (i > 0 && t <= obs[i - 1]) {
      set_error("b2m_loglik_stats: observation terms must be listed in increasing term order, each once");
      return 1;
    }
    if (!is_observation_term(m->terms[t], m->lin)) {
      set_error("b2m_loglik_stats: term " + std::to_string(t) + " is not an observation term (its value must be data or a "
                "constant and one of its distribution parameters must depend on the model parameters)");
      return 1;
    }
    obs[i] = t;
    total += m->terms[t].length;
  }
  if (total != n_obs) {
    set_error("b2m_loglik_stats: n_obs = " + std::to_string(n_obs) + " but the listed terms have " + std::to_string(total) +
              " observations");
    return 1;
  }
  int lik = -1;
  if (m->model_class == 1)
    for (int t = 0; t < n_terms; ++t) {
      const b2m_term &T = m->terms[t];
      if (T.x.kind == B2M_OP_MATVEC || T.p0.kind == B2M_OP_MATVEC || T.p1.kind == B2M_OP_MATVEC) lik = t;
    }
  B2M_MODEL_GUARD(m);
  return b2m::loglik_stats(m->km, m->model_class == 1 ? &m->glm : nullptr, lik, m->terms, obs, draws, n_draws, out, n_obs,
                           static_cast<cudaStream_t>(stream));
}

struct b2m_comm {
  b2m::Comm *c = nullptr;
};

int b2m_comm_unique_id(uint8_t *out128) {
  B2M_REQUIRE(out128 != nullptr, "b2m_comm_unique_id: NULL argument");
  return b2m::comm_unique_id(out128);
}

int b2m_comm_init(const uint8_t *id128, int32_t n_ranks, int32_t rank, b2m_comm **out) {
  B2M_REQUIRE(id128 && out, "b2m_comm_init: NULL argument");
  B2M_REQUIRE(n_ranks >= 1 && rank >= 0 && rank < n_ranks, "b2m_comm_init: rank out of range");
  *out = nullptr;
  b2m::Comm *c = nullptr;
  if (int rc = b2m::comm_init(id128, n_ranks, rank, &c)) return rc;
  *out = new b2m_comm{c};
  return 0;
}

void b2m_comm_destroy(b2m_comm *c) {
  if (!c) return;
  b2m::comm_destroy(c->c);
  delete c;
}

int b2m_model_set_comm(b2m_model *m, b2m_comm *c, void *stream) {
  B2M_REQUIRE(m != nullptr, "b2m_model_set_comm: NULL model");
  B2M_REQUIRE(m->model_class == 1, "b2m_model_set_comm: observation sharding is defined for GLM-class models (X @ beta) only");
  return b2m::glm_set_comm(m->glm, c ? c->c : nullptr, static_cast<cudaStream_t>(stream));
}

int b2m_comm_allreduce_f32(b2m_comm *c, float *buf, int64_t n, void *stream) {
  B2M_REQUIRE(c && buf && n >= 0, "b2m_comm_allreduce_f32: bad argument");
  return b2m::comm_allreduce_f32(c->c, buf, n, static_cast<cudaStream_t>(stream));
}

int b2m_peer_alloc(int64_t bytes, void **ptr, uint8_t *handle64) {
  B2M_REQUIRE(bytes > 0 && ptr && handle64, "b2m_peer_alloc: bad argument");
  return b2m::peer_alloc(bytes, ptr, handle64);
}
int b2m_peer_open(const uint8_t *handle64, void **ptr) {
  B2M_REQUIRE(handle64 && ptr, "b2m_peer_open: NULL argument");
  return b2m::peer_open(handle64, ptr);
}
int b2m_peer_close(void *ptr) { return ptr ? b2m::peer_close(ptr) : 0; }
int b2m_peer_free(void *ptr) { return ptr ? b2m::peer_free(ptr) : 0; }

int b2m_model_peer_bytes(b2m_model *m, int64_t n_chains, int32_t n_ranks, int64_t *bytes) {
  B2M_REQUIRE(m && bytes, "b2m_model_peer_bytes: NULL argument");
  B2M_REQUIRE(m->model_class == 1, "b2m_model_peer_bytes: the peer window is defined for GLM-class models only");
  B2M_REQUIRE(n_ranks >= 2 && n_ranks <= b2m::kMaxPeers, "b2m_model_peer_bytes: 2..8 ranks");
  B2M_REQUIRE(n_chains > 0 && n_chains % (128 * (int64_t)n_ranks) == 0 && n_chains % 256 == 0,
              "b2m_model_peer_bytes: n_chains must be a multiple of 256 and of 128 x the number of ranks");
  b2m::PeerWindow w;
  *bytes = (int64_t)b2m::peer_layout(w, n_chains, n_ranks, m->glm.Dp);
  return 0;
}

int b2m_model_peer_attach(b2m_model *m, void *const *windows, int32_t n_ranks, int32_t rank, int64_t n_chains, int64_t bytes) {
  B2M_REQUIRE(m && windows, "b2m_model_peer_attach: NULL argument");
  B2M_REQUIRE(m->model_class == 1, "b2m_model_peer_attach: the peer window is defined for GLM-class models only");
  B2M_REQUIRE(m->glm.lik == b2m::kLikNormal, "b2m_model_peer_attach: observation sharding is defined for the Normal likelihood only");
  B2M_REQUIRE(m->glm.use_tc == 2, "b2m_model_peer_attach: the peer exchange is built on the fp16-encoded tcgen05 path");
  B2M_REQUIRE(m->glm.tf == nullptr, "b2m_model_peer_attach: constraint transforms are not supported with the peer exchange");
  B2M_REQUIRE(n_ranks >= 2 && n_ranks <= b2m::kMaxPeers && rank >= 0 && rank < n_ranks, "b2m_model_peer_attach: 2..8 ranks");
  B2M_REQUIRE(n_chains > 0 && n_chains % (128 * (int64_t)n_ranks) == 0 && n_chains % 256 == 0,
              "b2m_model_peer_attach: n_chains must be a multiple of 256 and of 128 x the number of ranks");
  for (int s = 0; s < n_ranks; ++s) B2M_REQUIRE(windows[s] != nullptr, "b2m_model_peer_attach: NULL window");
  if (int rc = b2m::glm_use_streaming(m->glm, "the peer exchange of observation sharding")) return rc;
  return b2m::glm_peer_attach(m->glm, windows, n_ranks, rank, n_chains, bytes);
}

int b2m_mass_from_draws(const float *draws, int64_t S, int64_t C, int64_t D, float *inv_mass, void *stream) {
  B2M_REQUIRE(draws && inv_mass, "b2m_mass_from_draws: NULL argument");
  B2M_REQUIRE(S > 0 && C > 0 && D > 0, "b2m_mass_from_draws: sizes must be positive");
  return b2m::mass_from_draws(draws, S, C, D, inv_mass, static_cast<cudaStream_t>(stream));
}

int b2m_quantiles(const float *x, int64_t n, const double *q, int32_t n_q, double *out, void *stream) {
  B2M_REQUIRE(x && q && out, "b2m_quantiles: NULL argument");
  B2M_REQUIRE(n > 0 && n_q > 0 && n_q <= 8, "b2m_quantiles: need n > 0 and 1..8 quantiles");
  for (int i = 0; i < n_q; ++i) B2M_REQUIRE(q[i] >= 0.0 && q[i] <= 1.0, "b2m_quantiles: quantiles must lie in [0, 1]");
  return b2m::quantiles(x, n, q, n_q, out, static_cast<cudaStream_t>(stream));
}

int b2m_hmc_run(b2m_model *m, const b2m_hmc_args *a, void *stream) {
  B2M_REQUIRE(m && a, "b2m_hmc_run: NULL argument");
  B2M_REQUIRE(a->n_chains > 0 && a->n_iter >= 0 && a->n_leapfrog > 0, "b2m_hmc_run: bad sizes");
  B2M_REQUIRE(a->theta && a->step_size && a->n_accept && a->n_total, "b2m_hmc_run: NULL state pointer");
  B2M_REQUIRE(valid_lanes(a->lanes), "b2m_hmc_run: lanes must be 0 or a power of two <= 32");
  B2M_REQUIRE(a->adapt >= B2M_ADAPT_NONE && a->adapt <= B2M_ADAPT_DUAL_AVERAGING, "b2m_hmc_run: bad adapt mode");
  B2M_REQUIRE(a->adapt != B2M_ADAPT_DUAL_AVERAGING || a->da_state, "b2m_hmc_run: dual averaging needs da_state");
  if (a->n_iter == 0) return 0;
  B2M_MODEL_GUARD(m);
  if (m->model_class == 1) return b2m::glm_hmc_run(m->glm, *a, static_cast<cudaStream_t>(stream));
  return b2m::launch_hmc(m->km, *a, static_cast<cudaStream_t>(stream), m->jit);
}

int b2m_mh_run(b2m_model *m, const b2m_mh_args *a, void *stream) {
  B2M_REQUIRE(m && a, "b2m_mh_run: NULL argument");
  B2M_REQUIRE(a->n_chains > 0 && a->n_iter >= 0, "b2m_mh_run: bad sizes");
  B2M_REQUIRE(a->theta && a->logp && a->n_accept, "b2m_mh_run: NULL state pointer");
  B2M_REQUIRE(valid_lanes(a->lanes), "b2m_mh_run: lanes must be 0 or a power of two <= 32");
  if (a->n_iter == 0) return 0;
  B2M_MODEL_GUARD(m);
  if (m->model_class == 1) return b2m::glm_mh_run(m->glm, *a, static_cast<cudaStream_t>(stream));
  return b2m::launch_mh(m->km, *a, static_cast<cudaStream_t>(stream), m->jit);
}

int b2m_nuts_run(b2m_model *m, const b2m_nuts_args *a, void *stream) {
  B2M_REQUIRE(m && a, "b2m_nuts_run: NULL argument");
  B2M_REQUIRE(a->n_chains > 0 && a->n_iter >= 0, "b2m_nuts_run: bad sizes");
  B2M_REQUIRE(a->max_tree_depth >= 1 && a->max_tree_depth <= B2M_MAX_TREE_DEPTH, "b2m_nuts_run: max_tree_depth out of range");
  B2M_REQUIRE(a->theta && a->step_size && a->da_state && a->n_accept && a->n_leaves && a->n_diverge,
              "b2m_nuts_run: NULL state pointer");
  B2M_REQUIRE(valid_lanes(a->lanes), "b2m_nuts_run: lanes must be 0 or a power of two <= 32");
  B2M_REQUIRE(a->adapt == B2M_ADAPT_NONE || a->adapt == B2M_ADAPT_DUAL_AVERAGING || a->adapt == B2M_ADAPT_POOLED,
              "b2m_nuts_run: bad adapt mode");
  B2M_REQUIRE(a->adapt != B2M_ADAPT_POOLED || m->model_class == 1,
              "b2m_nuts_run: pooled step-size adaptation needs a GLM-class model (lock-step kernels)");
  B2M_REQUIRE(a->schedule == B2M_SCHED_ASYNC || a->schedule == B2M_SCHED_SYNC, "b2m_nuts_run: unknown schedule");
  B2M_REQUIRE(a->slice_state >= B2M_SLICE_OFF && a->slice_state <= B2M_SLICE_PEER, "b2m_nuts_run: unknown slice_state");
  B2M_REQUIRE(a->slice_state == B2M_SLICE_OFF || (m->model_class == 1 && m->glm.comm && a->adapt == B2M_ADAPT_NONE &&
                                                   a->schedule == B2M_SCHED_ASYNC),
              "b2m_nuts_run: slice_state needs an observation-sharded GLM-class model, the asynchronous schedule and no adaptation");
  if (a->n_iter == 0) return 0;
  B2M_MODEL_GUARD(m);
  if (m->model_class == 1) return b2m::glm_nuts_run(m->glm, *a, static_cast<cudaStream_t>(stream));
  return b2m::launch_nuts(m->km, *a, static_cast<cudaStream_t>(stream), m->jit);
}

}  // extern "C"

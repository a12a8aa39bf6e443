// Pointwise log-likelihood statistics over posterior draws (b2m_loglik_stats), reduced on the device.
//
//   ll[s, n] = w log p(x_n | params(theta_s))   for every draw s and every observation n of the listed terms
//   out[n] = (lppd_n, mean_n, var_n) = (log mean_s exp ll[s, n], mean_s ll[s, n], sample variance (ddof 1))
//
// The [S, N] matrix is never stored.  The draws are processed in batches of kLoglikBatch rows; per batch, every
// observation term writes partials of 32 draw rows each, (max, sum exp(ll - max), mean, M2) as float4
// [batch / 32, ld], and a fold kernel merges them in row order into a float64 running state [n_obs, 4] with Chan's
// parallel formulas.  Fixed batch size, fixed merge order: the result is bit-identical across calls.
//   * the X @ beta term of a GLM-class model: K5 with the statistics epilogue (glm.cu / glm_tc.cu)
//   * every other observation term: a SIMT kernel over (observation, 32-row group) with the operand fetchers and
//     densities of the pointwise class (model.cuh), theta read from the draw rows
#include <vector>

#include "glm.cuh"

namespace b2m {

constexpr int64_t kLoglikBatch = 4096;   // draw rows per batch (partials of the C4 term: 128 x 100K x 16 B)

__global__ void __launch_bounds__(128) loglik_pointwise_kernel(b2m_term T, const b2m_lin_entry *__restrict__ lin,
                                                               const DevArray *__restrict__ arrays,
                                                               const float *__restrict__ draws, int D, int64_t rows,
                                                               float4 *__restrict__ part) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= T.length) return;
  SModel sm;
  sm.terms = nullptr; sm.lin = lin; sm.arrays = arrays; sm.n_terms = 0; sm.D = D;
  const int64_t row0 = (int64_t)blockIdx.y * 32, left = rows - row0;
  const int nv = left >= 32 ? 32 : (int)left;
  float ll[32];
  float mx = -INFINITY, s = 0.f;
#pragma unroll
  for (int r = 0; r < 32; ++r) {
    ll[r] = 0.f;
    if (r < nv) {
      const float *th = draws + (row0 + r) * D;
      const float x = op_fetch(T.x, n, th, 1, sm), p0 = op_fetch(T.p0, n, th, 1, sm), p1 = op_fetch(T.p1, n, th, 1, sm);
      ll[r] = dist_eval<false>(T.dist, x, p0, p1, T.k0, T.k1, T.k2).lp * T.weight;
      mx = fmaxf(mx, ll[r]);
      s += ll[r];
    }
  }
  const float mean = s / (float)nv;
  float se = 0.f, m2 = 0.f;
#pragma unroll
  for (int r = 0; r < 32; ++r)
    if (r < nv) {
      se += mx == -INFINITY ? 0.f : expf(ll[r] - mx);
      const float d = ll[r] - mean;
      m2 = fmaf(d, d, m2);
    }
  part[blockIdx.y * (int64_t)T.length + n] = make_float4(mx, se, mean, m2);
}

// state[n] = (max, sum exp(ll - max), mean, M2) over the `done` draws before this batch, merged with the partials of the
// batch's `rows` draws, group by group in row order
__global__ void __launch_bounds__(256) loglik_fold_kernel(const float4 *__restrict__ part, int64_t ld, int n_cols,
                                                          int64_t rows, int64_t done, double *__restrict__ state) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= n_cols) return;
  double *st = state + (int64_t)n * 4;
  double m = -INFINITY, se = 0.0, mean = 0.0, m2 = 0.0;
  if (done > 0) { m = st[0]; se = st[1]; mean = st[2]; m2 = st[3]; }
  double cnt = (double)done;
  const int64_t groups = (rows + 31) / 32;
  for (int64_t gi = 0; gi < groups; ++gi) {
    const float4 p = part[gi * ld + n];
    const int64_t left = rows - gi * 32;
    const double nb = (double)(left >= 32 ? 32 : left);
    const double pm = (double)p.x;
    const double mm = pm > m ? pm : m;
    if (mm != -INFINITY)
      se = (m == -INFINITY ? 0.0 : se * exp(m - mm)) + (pm == -INFINITY ? 0.0 : (double)p.y * exp(pm - mm));
    m = mm;
    const double tot = cnt + nb, delta = (double)p.z - mean;
    mean += delta * (nb / tot);
    m2 += (double)p.w + delta * delta * (cnt * nb / tot);
    cnt = tot;
  }
  st[0] = m; st[1] = se; st[2] = mean; st[3] = m2;
}

__global__ void loglik_finalize_kernel(const double *__restrict__ state, int64_t n_obs, int64_t S, double *__restrict__ out) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= n_obs) return;
  const double *st = state + n * 4;
  out[n * 3 + 0] = st[0] + log(st[1]) - log((double)S);
  out[n * 3 + 1] = st[2];
  out[n * 3 + 2] = S > 1 ? st[3] / (double)(S - 1) : 0.0;
}

static int fold(const float4 *part, int64_t ld, int n_cols, int64_t rows, int64_t done, double *state, cudaStream_t st) {
  loglik_fold_kernel<<<(n_cols + 255) / 256, 256, 0, st>>>(part, ld, n_cols, rows, done, state);
  ++g_launches;
  B2M_CHECK_CUDA(cudaGetLastError());
  return 0;
}

// `obs` = the observation terms (indices into `terms`, increasing), `lik` = index of the X @ beta term of a GLM-class
// model (g != nullptr) or -1.  The caller has validated the arguments.
int loglik_stats(const KModel &km, GlmModel *g, int lik, const std::vector<b2m_term> &terms, const std::vector<int> &obs,
                 const float *draws, int64_t S, double *out, int64_t n_obs, cudaStream_t st) {
  const int D = km.D;
  int64_t ld_max = 1;
  std::vector<int64_t> off(obs.size());
  int64_t o = 0;
  bool glm_term = false;
  for (size_t i = 0; i < obs.size(); ++i) {
    off[i] = o;
    o += terms[obs[i]].length;
    const bool mv = g && obs[i] == lik;
    glm_term = glm_term || mv;
    const int64_t ld = mv ? g->Np : terms[obs[i]].length;
    if (ld > ld_max) ld_max = ld;
  }
  const int64_t B = S < kLoglikBatch ? S : kLoglikBatch;
  const int64_t groups = (B <= 128 ? 128 : (B + 255) / 256 * 256) / 32;   // whole tiles of the K5 batch
  float4 *part = nullptr;
  double *state = nullptr;
  B2M_CHECK_CUDA(cudaMallocAsync(reinterpret_cast<void **>(&part), sizeof(float4) * groups * ld_max, st));
  int rc = cudaMallocAsync(reinterpret_cast<void **>(&state), sizeof(double) * 4 * (n_obs > 0 ? n_obs : 1), st) == cudaSuccess ? 0 : 2;
  if (rc) set_error("b2m_loglik_stats: out of device memory for the running state");
  if (!rc && glm_term) rc = glm_loglik_center(*g, draws, S, st);
  for (int64_t b0 = 0; b0 < S && !rc; b0 += B) {
    const int64_t rows = S - b0 < B ? S - b0 : B;
    const float *batch = draws + b0 * D;
    for (size_t i = 0; i < obs.size() && !rc; ++i) {
      const b2m_term &T = terms[obs[i]];
      if (g && obs[i] == lik) {
        rc = glm_loglik_batch(*g, batch, rows, part, st);
        if (!rc) rc = fold(part, g->Np, g->N, rows, b0, state + off[i] * 4, st);
      } else {
        loglik_pointwise_kernel<<<dim3((unsigned)((T.length + 127) / 128), (unsigned)((rows + 31) / 32)), 128, 0, st>>>(
            T, km.lin, km.arrays, batch, D, rows, part);
        ++g_launches;
        if (cudaGetLastError() != cudaSuccess) { set_error("b2m_loglik_stats: pointwise kernel launch failed"); rc = 2; }
        if (!rc) rc = fold(part, T.length, T.length, rows, b0, state + off[i] * 4, st);
      }
    }
  }
  if (!rc) {
    loglik_finalize_kernel<<<(unsigned)((n_obs + 255) / 256), 256, 0, st>>>(state, n_obs, S, out);
    ++g_launches;
    if (cudaGetLastError() != cudaSuccess) { set_error("b2m_loglik_stats: finalize launch failed"); rc = 2; }
  }
  if (state) cudaFreeAsync(state, st);
  cudaFreeAsync(part, st);
  return rc;
}

}  // namespace b2m

// GLM-class evaluation pipeline: pack -> GEMM (B X^T) with residual epilogue -> GEMM (R X) -> finish.
#include "glm_rows.cuh"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

namespace b2m {

// ---------------------------------------------------------------- memory
template <typename T>
static int dev_alloc(T **p, size_t n) {
  B2M_CHECK_CUDA(cudaMalloc(reinterpret_cast<void **>(p), sizeof(T) * (n ? n : 1)));
  return 0;
}
#define FREE(p) do { if (p) cudaFree(p); p = nullptr; } while (0)

static void free_workspace(GlmModel &g) {
  FREE(g.B); FREE(g.Bh); FREE(g.Bl); FREE(g.R); FREE(g.Rh); FREE(g.Rl); FREE(g.G); FREE(g.ss_part); FREE(g.inv_var);
  FREE(g.red); FREE(g.B16h); FREE(g.B16l); FREE(g.R16h); FREE(g.R16l); FREE(g.a_unscale); FREE(g.r_scale); FREE(g.r_unscale);
  FREE(g.thc);
  g.cap = 0;
}

void glm_free(GlmModel &g) {
  free_workspace(g);
  FREE(g.X); FREE(g.XT); FREE(g.Xh); FREE(g.Xl); FREE(g.XTh); FREE(g.XTl); FREE(g.y);
  FREE(g.y0); FREE(g.beta0); FREE(g.center_part);
  FREE(g.X16h); FREE(g.X16l); FREE(g.XT16h); FREE(g.XT16l); FREE(g.col_scale); FREE(g.inv_col_scale); FREE(g.y0max_bits);
  FREE(g.colmax);
  FREE(g.G64); FREE(g.gvec); FREE(g.gb); FREE(g.gterm); FREE(g.Gmh); FREE(g.Gml); FREE(g.g_unscale);
  FREE(g.ws);
  FREE(g.tf); FREE(g.blk_counter);
  g.ws_cap = 0;
  if (g.h_flag) cudaFreeHost(g.h_flag);
  g.h_flag = nullptr;
  if (g.h_prog) cudaFreeHost(const_cast<long long *>(g.h_prog));
  g.h_prog = nullptr;
}

int glm_reserve(GlmModel &g, int64_t n_chains) {
  const int64_t cp = (n_chains + 255) / 256 * 256;   // whole CTA-pair tiles (glm_tc.cu)
  if (cp <= g.cap) return 0;
  free_workspace(g);
  // split-K partials: a compacted batch of fewer rows may use more splits -- size G for the worst case
  size_t g_rows = (size_t)cp;
  if (g.use_tc)
    for (int64_t c = 128; c <= cp; c += 128) {
      const size_t need = (size_t)contraction_splits(g, c) * (size_t)c;
      if (need > g_rows) g_rows = need;
    }
  g.g_splits_cap = (int)((g_rows + cp - 1) / cp);
  if (dev_alloc(&g.B, cp * g.Dp) || dev_alloc(&g.G, g_rows * g.Dp) || dev_alloc(&g.inv_var, cp) ||
      dev_alloc(&g.red, (size_t)cp * g.Dp + cp))
    return 2;
  if (g.tf && dev_alloc(&g.thc, (size_t)cp * g.Dtot)) return 2;
  // the residual operand R [cap, Np] and the per-tile sums exist only in the streaming form (2 x 1.6 GB at C4 in fp16)
  const bool stream = g.form == kFormStream;
  if (stream && dev_alloc(&g.ss_part, (size_t)(g.Np / 64) * cp)) return 2;
  if (g.use_tc == 0 && dev_alloc(&g.R, cp * (size_t)g.Np)) return 2;
  if (g.use_tc == 1) {
    if (dev_alloc(&g.Bh, cp * g.Dp) || dev_alloc(&g.Bl, cp * g.Dp)) return 2;
    if (stream && (dev_alloc(&g.Rh, cp * (size_t)g.Np) || dev_alloc(&g.Rl, cp * (size_t)g.Np))) return 2;
  }
  if (g.use_tc == 2) {
    if (dev_alloc(&g.B16h, cp * g.Dp) || dev_alloc(&g.B16l, cp * g.Dp) || dev_alloc(&g.a_unscale, cp)) return 2;
    if (stream && (dev_alloc(&g.R16h, cp * (size_t)g.Np) || dev_alloc(&g.R16l, cp * (size_t)g.Np) ||
                   dev_alloc(&g.r_scale, cp) || dev_alloc(&g.r_unscale, cp)))
      return 2;
  }
  g.cap = cp;
  return 0;
}

// ---------------------------------------------------------------- data preparation (once per model)
__global__ void pad_transpose_kernel(const float *__restrict__ X, int N, int D, int Np, int Dp, float *Xp, float *XT) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)Np * Dp) return;
  const int n = int(i / Dp), d = int(i % Dp);
  const float v = (n < N && d < D) ? X[(int64_t)n * D + d] : 0.f;
  Xp[i] = v;
  if (XT) XT[(int64_t)d * Np + n] = v;
}

__global__ void split_tf32_kernel(const float *__restrict__ Xp, int Np, int Dp, float *Xh, float *Xl, float *XTh, float *XTl) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)Np * Dp) return;
  const int n = int(i / Dp), d = int(i % Dp);
  float hi, lo;
  split_tf32(Xp[i], hi, lo);
  Xh[i] = hi; Xl[i] = lo;
  XTh[(int64_t)d * Np + n] = hi; XTl[(int64_t)d * Np + n] = lo;
}

__global__ void pad_vector_kernel(const float *__restrict__ y, int N, int Np, float *yp) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < Np) yp[i] = i < N ? y[i] : 0.f;
}

// fp16 encoding: column maxima and the largest row norm of the padded X
__global__ void __launch_bounds__(256) x_stats_kernel(const float *__restrict__ Xp, int Np, int Dp, unsigned *colmax_bits,
                                                      unsigned *rownorm_bits) {
  // block (32, 8): 32 columns x 8 row lanes, rows strided by gridDim.y * 8
  const int d = blockIdx.x * 32 + threadIdx.x;
  float cm = 0.f;
  for (int n = blockIdx.y * 8 + threadIdx.y; n < Np; n += gridDim.y * 8) cm = fmaxf(cm, fabsf(Xp[(int64_t)n * Dp + d]));
  atomicMax(colmax_bits + d, __float_as_uint(cm));   // non-negative floats order like their bit patterns
  if (blockIdx.x == 0) {                             // row norms: one warp (threadIdx.y) per row, lanes stride the columns
    for (int n = blockIdx.y * 8 + threadIdx.y; n < Np; n += gridDim.y * 8) {
      float s = 0.f;
      for (int c = threadIdx.x; c < Dp; c += 32) { const float v = Xp[(int64_t)n * Dp + c]; s = fmaf(v, v, s); }
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (threadIdx.x == 0) atomicMax(rownorm_bits, __float_as_uint(sqrtf(s)));
    }
  }
}

// Entries of a column below its maximum x 2^-17 land, after the column is scaled to just under 2^14, where the lo half
// of the fp16 split is subnormal: they keep fewer than the nominal 22 bits.  Count them (zeros are exact and excluded).
__global__ void __launch_bounds__(256) x_small_count_kernel(const float *__restrict__ Xp, int Np, int Dp,
                                                            const unsigned *__restrict__ colmax_bits, unsigned *small) {
  const int d = blockIdx.x * 32 + threadIdx.x;
  const float thr = __uint_as_float(colmax_bits[d]) * 7.62939453125e-6f;   // 2^-17
  unsigned cnt = 0;
  for (int n = blockIdx.y * 8 + threadIdx.y; n < Np; n += gridDim.y * 8) {
    const float a = fabsf(Xp[(int64_t)n * Dp + d]);
    cnt += (a > 0.f && a < thr) ? 1u : 0u;
  }
  if (cnt) atomicAdd(small + d, cnt);
}

__global__ void col_scale_kernel(const unsigned *__restrict__ colmax_bits, int Dp, float *col_scale, float *inv_col_scale,
                                 float *colmax) {
  const int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= Dp) return;
  const float m = __uint_as_float(colmax_bits[d]);
  const float s = pow2_scale(m);
  col_scale[d] = s;
  inv_col_scale[d] = 1.0f / s;
  if (colmax) colmax[d] = m;
}

__global__ void split_f16_kernel(const float *__restrict__ Xp, int Np, int Dp, const float *__restrict__ col_scale,
                                 __half *Xh, __half *Xl, __half *XTh, __half *XTl) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)Np * Dp) return;
  const int n = int(i / Dp), d = int(i % Dp);
  __half hi, lo;
  split_f16(Xp[i] * col_scale[d], hi, lo);
  Xh[i] = hi; Xl[i] = lo;
  XTh[(int64_t)d * Np + n] = hi; XTl[(int64_t)d * Np + n] = lo;
}

// labels of a Bernoulli likelihood: count the entries of y[0, N) that are neither 0 nor 1 (NaN included)
__global__ void count_bad_labels_kernel(const float *__restrict__ y, int N, unsigned *bad) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const bool b = i < N && !(y[i] == 0.f || y[i] == 1.f);
  const unsigned n = __popc(__ballot_sync(0xffffffffu, b));
  if ((threadIdx.x & 31) == 0 && n) atomicAdd(bad, n);
}

int glm_check_labels(const float *y, int N) {
  unsigned *d = nullptr, h = 0;
  B2M_CHECK_CUDA(cudaMalloc(&d, sizeof(unsigned)));
  B2M_CHECK_CUDA(cudaMemset(d, 0, sizeof(unsigned)));
  if (N > 0) count_bad_labels_kernel<<<(N + 255) / 256, 256>>>(y, N, d);
  ++g_launches;
  const cudaError_t e = cudaMemcpy(&h, d, sizeof(unsigned), cudaMemcpyDeviceToHost);
  cudaFree(d);
  B2M_CHECK_CUDA(e);
  if (h) {
    set_error("GLM class: Bernoulli labels must all be 0 or 1 (" + std::to_string(h) + " of " + std::to_string(N) +
              " are not)");
    return 1;
  }
  return 0;
}

// ---------------------------------------------------------------- Gram form: statistics (once per model)
// Gram matrix of the augmented matrix A = [X | y | 1 | 0 ...] ([Np, Da], Da = Dp + 64): column Dp is y, column Dp + 1
// the indicator of the N real rows, so one pass yields X^T X, X^T y, X^T 1, ||y||^2 and sum y.  Products of fp32 values
// are exact in float64; only the sums round.  Upper-triangle 64 x 64 tiles (blockIdx.x), each over one slice of the
// rows (blockIdx.y); the slices are added in a fixed order afterwards.
constexpr int GT = 64, GK = 16;

__device__ __forceinline__ double aug_at(const float *__restrict__ X, const float *__restrict__ y, int N, int Dp, int n, int d) {
  if (d < Dp) return (double)X[(int64_t)n * Dp + d];
  if (d == Dp) return (double)y[n];   // padding rows of y are 0
  return (d == Dp + 1 && n < N) ? 1.0 : 0.0;
}

__global__ void __launch_bounds__(256) gram_partial_kernel(const float *__restrict__ X, const float *__restrict__ y, int N,
                                                           int Np, int Dp, int Da, int rows_per_slice, double *__restrict__ part) {
  __shared__ double sA[GK][GT], sB[GK][GT];
  const int nt = Da / GT;
  int t = blockIdx.x, ti = 0;
  while (t >= nt - ti) { t -= nt - ti; ++ti; }
  const int i0 = ti * GT, j0 = (ti + t) * GT;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int n_begin = blockIdx.y * rows_per_slice, n_end = min(n_begin + rows_per_slice, Np);
  double acc[4][4] = {};
  for (int n0 = n_begin; n0 < n_end; n0 += GK) {
    for (int e = threadIdx.x; e < GK * GT; e += 256) {
      const int r = e / GT, col = e % GT, n = n0 + r;
      sA[r][col] = n < n_end ? aug_at(X, y, N, Dp, n, i0 + col) : 0.0;
      sB[r][col] = n < n_end ? aug_at(X, y, N, Dp, n, j0 + col) : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < GK; ++k) {
      double a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = sA[k][ty + 16 * i]; b[i] = sB[k][tx + 16 * i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fma(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j)
      part[((size_t)blockIdx.y * Da + i0 + ty + 16 * i) * Da + j0 + tx + 16 * j] = acc[i][j];
}

// G64 (mirrored from the upper tiles: a diagonal tile computes (i, j) and (j, i) from the same products in the same
// order, so G64 is exactly symmetric) and gvec = X^T y || X^T 1 || ||y||^2 || sum y
__global__ void gram_final_kernel(const double *__restrict__ part, int S, int Da, int Dp, double *__restrict__ G64,
                                  double *__restrict__ gvec) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nG = (int64_t)Dp * Dp;
  if (i >= nG + 2 * Dp + 2) return;
  int r, c;
  if (i < nG) { r = int(i / Dp); c = int(i % Dp); }
  else {
    const int k = int(i - nG);
    if (k < Dp) { r = k; c = Dp; }
    else if (k < 2 * Dp) { r = k - Dp; c = Dp + 1; }
    else { r = Dp; c = k == 2 * Dp ? Dp : Dp + 1; }
  }
  if (r / GT > c / GT) { const int tmp = r; r = c; c = tmp; }
  double s = 0.0;
  for (int z = 0; z < S; ++z) s += part[((size_t)z * Da + r) * Da + c];
  if (i < nG) G64[i] = s; else gvec[i - nG] = s;
}

// B operand of the per-leaf contraction, one block per column j of G~ = diag(cs) G diag(cs) (cs = col_scale of the fp16
// encoding, 1 for tf32).  fp16: column j is scaled by the power of two t_j that puts its maximum just below 2^14 (the
// entries reach N max|x|^2 otherwise), then split into hi / lo halves; row j of the stored operand = column j (K-major).
__global__ void __launch_bounds__(256) gram_operand_kernel(const double *__restrict__ G64, int Dp,
                                                           const float *__restrict__ col_scale, void *Gh, void *Gl,
                                                           float *__restrict__ g_unscale) {
  __shared__ double red[256];
  const int j = blockIdx.x;
  const double csj = col_scale ? (double)col_scale[j] : 1.0;
  double m = 0.0;
  for (int k = threadIdx.x; k < Dp; k += 256) {
    const double ck = col_scale ? (double)col_scale[k] : 1.0;
    m = fmax(m, fabs(ck * G64[(int64_t)k * Dp + j] * csj));
  }
  red[threadIdx.x] = m;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] = fmax(red[threadIdx.x], red[threadIdx.x + o]);
    __syncthreads();
  }
  const double t = col_scale ? (double)pow2_scale((float)red[0]) : 1.0;
  for (int k = threadIdx.x; k < Dp; k += 256) {
    const double ck = col_scale ? (double)col_scale[k] : 1.0;
    const double v = ck * G64[(int64_t)k * Dp + j] * csj * t;   // powers of two: exact
    const int64_t o = (int64_t)j * Dp + k;
    if (col_scale) {
      const __half hi = __double2half(v);
      static_cast<__half *>(Gh)[o] = hi;
      static_cast<__half *>(Gl)[o] = __double2half(v - (double)__half2float(hi));
    } else {
      float hi, lo;
      split_tf32((float)v, hi, lo);
      static_cast<float *>(Gh)[o] = hi;
      static_cast<float *>(Gl)[o] = lo;
    }
  }
  if (threadIdx.x == 0 && g_unscale) g_unscale[j] = (float)(1.0 / (csj * t));
}

static int gram_build(GlmModel &g) {
  const int Dp = g.Dp, Da = Dp + GT;
  const size_t dd = (size_t)Dp * Dp;
  const bool f16 = g.use_tc == 2;
  if (dev_alloc(&g.G64, dd) || dev_alloc(&g.gvec, 2 * (size_t)Dp + 2) || dev_alloc(&g.gb, (size_t)Dp + 1) ||
      dev_alloc(&g.gterm, Dp))
    return 2;
  B2M_CHECK_CUDA(cudaMalloc(&g.Gmh, dd * (f16 ? 2 : 4)));
  B2M_CHECK_CUDA(cudaMalloc(&g.Gml, dd * (f16 ? 2 : 4)));
  if (f16 && dev_alloc(&g.g_unscale, Dp)) return 2;
  // row slices: about two blocks per SM in all, each slice a whole number of 256-row blocks
  const int nt = Da / GT, tiles = nt * (nt + 1) / 2;
  int S = (296 + tiles - 1) / tiles;
  if (S > g.Np / 256) S = g.Np / 256;
  if (S < 1) S = 1;
  const int rows_per_slice = (g.Np / 256 + S - 1) / S * 256;
  S = (g.Np + rows_per_slice - 1) / rows_per_slice;
  double *part = nullptr;
  if (dev_alloc(&part, (size_t)S * Da * Da)) return 2;
  gram_partial_kernel<<<dim3((unsigned)tiles, (unsigned)S), 256>>>(g.X, g.y, g.N, g.Np, Dp, Da, rows_per_slice, part);
  const int64_t nf = (int64_t)dd + 2 * Dp + 2;
  gram_final_kernel<<<(unsigned)((nf + 255) / 256), 256>>>(part, S, Da, Dp, g.G64, g.gvec);
  gram_operand_kernel<<<Dp, 256>>>(g.G64, Dp, f16 ? g.col_scale : nullptr, g.Gmh, g.Gml, g.g_unscale);
  g_launches += 3;
  B2M_CHECK_CUDA(cudaGetLastError());
  const cudaError_t e = cudaDeviceSynchronize();
  cudaFree(part);
  B2M_CHECK_CUDA(e);
  return 0;
}

// b2m_model_options.glm_form -> GlmModel::form.  Auto: the Gram form for the Normal likelihood on a tensor-core path when
// N >= 2 Dp (the per-leaf contraction is then at most a quarter of the streaming form's flops) and Dp <= kGramMaxDp
// (the Gram arrays stay small).  Observation sharding switches back later (glm_use_streaming).
static int resolve_form(GlmModel &g) {
  if (g.form_req == kFormStream) { g.form = kFormStream; return 0; }
  const bool possible = g.lik == kLikNormal && g.use_tc != 0;
  if (g.form_req == kFormGram) {
    B2M_REQUIRE(g.lik == kLikNormal, "glm_form = gram: the Gram form is defined for the Normal likelihood only (the "
                                     "Bernoulli-logit likelihood has no closed form in X^T X); use 'auto' or 'stream'");
    B2M_REQUIRE(g.use_tc != 0, "glm_form = gram: the Gram form runs on the tensor-core paths (glm_path 'tc' / 'tc16'), "
                               "the SIMT path keeps the streaming form");
    g.form = kFormGram;
    return 0;
  }
  g.form = (possible && (int64_t)g.N >= 2 * (int64_t)g.Dp && g.Dp <= kGramMaxDp) ? kFormGram : kFormStream;
  return 0;
}

int glm_use_streaming(GlmModel &g, const char *why) {
  if (g.form == kFormStream) return 0;
  if (g.form_req == kFormGram) {
    set_error(std::string("glm_form = gram: ") + why + " needs the streaming form (create the model with glm_form 'auto' or 'stream')");
    return 1;
  }
  g.form = kFormStream;
  free_workspace(g);   // the next reservation allocates the residual operand of the streaming form
  return 0;
}

int glm_build(GlmModel &g, const float *X, const float *y, int N, int D, bool force_tc16) {
  g.N = N; g.D = D;
  g.N_total = N;
  g.Np = (N + 255) / 256 * 256;
  g.Dp = (D + 63) / 64 * 64;
  const size_t nd = (size_t)g.Np * g.Dp;
  if (dev_alloc(&g.X, nd) || dev_alloc(&g.y, g.Np) || dev_alloc(&g.y0, g.Np) || dev_alloc(&g.beta0, g.Dp) ||
      dev_alloc(&g.center_part, (size_t)kCenterSlices * g.Dp) || dev_alloc(&g.y0max_bits, 1))
    return 2;
  if (g.use_tc == 0 && dev_alloc(&g.XT, nd)) return 2;
  pad_transpose_kernel<<<(unsigned)((nd + 255) / 256), 256>>>(X, N, D, g.Np, g.Dp, g.X, g.XT);
  pad_vector_kernel<<<(g.Np + 255) / 256, 256>>>(y, N, g.Np, g.y);
  g_launches += 2;
  if (g.use_tc == 2) {
    // column maxima and the largest row norm; then, per column, how many entries are so far below the column's
    // maximum (< 2^-17 of it) that the scaled fp16 split cannot hold them to full precision: data with more than
    // 0.1 % of such entries in some column (one wild outlier is enough) keeps the tf32 encoding (8-bit exponent)
    unsigned *stats = nullptr;   // [Dp] column maxima (float bits) + [1] largest row norm + [Dp] small-entry counts
    if (dev_alloc(&stats, 2 * g.Dp + 1)) return 2;
    B2M_CHECK_CUDA(cudaMemset(stats, 0, sizeof(unsigned) * (2 * g.Dp + 1)));
    x_stats_kernel<<<dim3(g.Dp / 32, 64), dim3(32, 8)>>>(g.X, g.Np, g.Dp, stats, stats + g.Dp);
    x_small_count_kernel<<<dim3(g.Dp / 32, 64), dim3(32, 8)>>>(g.X, g.Np, g.Dp, stats, stats + g.Dp + 1);
    g_launches += 2;
    std::vector<unsigned> hmax(2 * g.Dp + 1);
    B2M_CHECK_CUDA(cudaMemcpy(hmax.data(), stats, sizeof(unsigned) * (2 * g.Dp + 1), cudaMemcpyDeviceToHost));
    memcpy(&g.x_rownorm_max, &hmax[g.Dp], sizeof(float));
    bool ok = g.x_rownorm_max < 3.0e38f;
    for (int d = 0; d < g.Dp && ok; ++d) {
      float m;
      memcpy(&m, &hmax[d], sizeof(float));
      if (!(m < 3.0e38f)) ok = false;                                  // inf / NaN in the data
      if ((double)hmax[g.Dp + 1 + d] > 1e-3 * (double)(N > 0 ? N : 1)) ok = false;
    }
    if (!ok && !force_tc16) g.use_tc = 1;   // wide-range data: tf32 encoding
    if (g.use_tc == 2) {
      if (dev_alloc(&g.X16h, nd) || dev_alloc(&g.X16l, nd) || dev_alloc(&g.XT16h, nd) || dev_alloc(&g.XT16l, nd) ||
          dev_alloc(&g.col_scale, g.Dp) || dev_alloc(&g.inv_col_scale, g.Dp) || dev_alloc(&g.colmax, g.Dp))
        return 2;
      col_scale_kernel<<<(g.Dp + 127) / 128, 128>>>(stats, g.Dp, g.col_scale, g.inv_col_scale, g.colmax);
      split_f16_kernel<<<(unsigned)((nd + 255) / 256), 256>>>(g.X, g.Np, g.Dp, g.col_scale, g.X16h, g.X16l, g.XT16h, g.XT16l);
      g_launches += 2;
    }
    B2M_CHECK_CUDA(cudaDeviceSynchronize());
    cudaFree(stats);
  }
  if (g.use_tc == 1) {
    if (dev_alloc(&g.Xh, nd) || dev_alloc(&g.Xl, nd) || dev_alloc(&g.XTh, nd) || dev_alloc(&g.XTl, nd)) return 2;
    split_tf32_kernel<<<(unsigned)((nd + 255) / 256), 256>>>(g.X, g.Np, g.Dp, g.Xh, g.Xl, g.XTh, g.XTl);
    ++g_launches;
  }
  B2M_CHECK_CUDA(cudaGetLastError());
  B2M_CHECK_CUDA(cudaDeviceSynchronize());
  if (int rc = resolve_form(g)) return rc;   // after the encoding is final (the Gram operand uses its column scales)
  if (g.form == kFormGram) return gram_build(g);
  return 0;
}

// ---------------------------------------------------------------- centering (once per sampler iteration)
// Near the posterior mode the residual z = y - X beta is a small difference of large numbers, and the gradient
// X^T z amplifies any systematic error of X beta by N (the tensor core accumulates with truncation: measured
// 1e-6 relative shrinkage of X beta => 1e-6 * N * |beta| absolute error in the gradient).  The contraction is
// therefore taken around a reference point beta0 shared by all chains of the batch:
//     z_c = (y - c - X beta0) - X (beta_c - beta0)
// with y0 = y - c - X beta0 accumulated in float64 once per sampler iteration (one GEMV, X read once) and
// beta0 = the mean of the chains' current positions.  X (beta_c - beta0) is then of the size of the
// posterior spread, and its rounding no longer dominates z.  Same function, different association.

// `tf` (sampler coordinates, nullptr otherwise): the centre is the mean of the constrained coefficients T(theta)_beta,
// the values that pack subtracts beta0 from -- so that delta stays of the size of the posterior spread when beta itself
// is transformed, and the samplers' centring agrees with that of the draws (glm_loglik_center).
__global__ void __launch_bounds__(256) glm_center_partial_kernel(const float *__restrict__ theta, const int *__restrict__ tf,
                                                                 int64_t C, int Dtot, int beta_off, int D, int Dp,
                                                                 double *__restrict__ part) {
  __shared__ double sh[8][33];
  const int d = blockIdx.x * 32 + threadIdx.x, ty = threadIdx.y;
  const int64_t per = (C + kCenterSlices - 1) / kCenterSlices;
  const int64_t c0 = (int64_t)blockIdx.y * per, c1 = (c0 + per < C) ? c0 + per : C;
  double acc = 0.0;
  if (d < D)
    for (int64_t c = c0 + ty; c < c1; c += 8) {
      float v = theta[c * Dtot + beta_off + d];
      if (tf) v = tf_constrain(tf[beta_off + d], v);
      if (fabsf(v) <= 3.0e38f) acc += (double)v;   // a diverged / NaN chain must not move the centre
    }
  sh[ty][threadIdx.x] = acc;
  __syncthreads();
  if (ty == 0) {
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += sh[i][threadIdx.x];   // fixed order => deterministic
    part[(int64_t)blockIdx.y * Dp + d] = s;
  }
}

__global__ void glm_center_final_kernel(const double *__restrict__ part, int Dp, int64_t C, float *__restrict__ beta0) {
  const int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= Dp) return;
  double s = 0.0;
  for (int i = 0; i < kCenterSlices; ++i) s += part[(int64_t)i * Dp + d];
  beta0[d] = (float)(s / (double)C);
}

// y0[n] = (y[n] - c) - sum_d X[n, d] beta0[d], float64 accumulation, one warp per observation row.
// logit: y0[n] = eta0[n] = c + sum_d X[n, d] beta0[d] instead (padding rows: -inf, see GlmModel::y0).
__global__ void __launch_bounds__(256) glm_y0_kernel(const float *__restrict__ X, const float *__restrict__ y,
                                                     const float *__restrict__ beta0, int N, int Np, int Dp,
                                                     float loc_const, float *__restrict__ y0,
                                                     unsigned *__restrict__ y0max_bits, bool logit) {
  extern __shared__ float sb[];
  for (int d = threadIdx.x; d < Dp; d += blockDim.x) sb[d] = beta0[d];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int n = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (n >= Np) return;
  double acc = 0.0;
  if (n < N) {
    const float4 *row = reinterpret_cast<const float4 *>(X + (int64_t)n * Dp);
    const float4 *b4 = reinterpret_cast<const float4 *>(sb);
    for (int i = lane; i < Dp / 4; i += 32) {
      const float4 x = __ldg(row + i), b = b4[i];
      acc += (double)x.x * b.x + (double)x.y * b.y + (double)x.z * b.z + (double)x.w * b.w;
    }
  }
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) {
    if (logit) {
      y0[n] = n < N ? (float)((double)loc_const + acc) : -INFINITY;
    } else {
      const float v = n < N ? (float)(((double)y[n] - (double)loc_const) - acc) : 0.f;
      y0[n] = v;
      if (v == v) atomicMax(y0max_bits, __float_as_uint(fabsf(v)));
    }
  }
}

// Gram form: the same centring from the build-time statistics, without reading X (O(Dp^2), float64):
//     b = X^T y0 = (v - c s1) - G beta0                                 v = X^T y, s1 = X^T 1
//     q = ||y0||^2 = ||y||^2 - 2 c sum y + N c^2 - beta0 . (2 (v - c s1) - G beta0)
// q is a difference of large numbers (||y||^2 ~ 1e8 against q ~ 1e5 at C4): harmless in float64, not in float32.
// One warp per coefficient d: b_d and the term beta0_d (2 (v_d - c s1_d) - (G beta0)_d) of q.
__global__ void __launch_bounds__(256) gram_center_kernel(const double *__restrict__ G64, const double *__restrict__ gvec,
                                                          const float *__restrict__ beta0, int Dp, float loc_const,
                                                          double *__restrict__ gb, double *__restrict__ gterm) {
  const int lane = threadIdx.x & 31;
  const int d = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (d >= Dp) return;
  double u = 0.0;
  for (int k = lane; k < Dp; k += 32) u = fma(G64[(int64_t)d * Dp + k], (double)beta0[k], u);
  for (int o = 16; o > 0; o >>= 1) u += __shfl_xor_sync(0xffffffffu, u, o);
  if (lane == 0) {
    const double w = gvec[d] - (double)loc_const * gvec[Dp + d];
    gb[d] = w - u;
    gterm[d] = (double)beta0[d] * (2.0 * w - u);
  }
}

// q = gb[Dp], one block, fixed summation order
__global__ void __launch_bounds__(256) gram_q_kernel(const double *__restrict__ gvec, const double *__restrict__ gterm,
                                                     int Dp, int N, float loc_const, double *__restrict__ gb) {
  __shared__ double sh[256];
  double s = 0.0;
  for (int d = threadIdx.x; d < Dp; d += 256) s += gterm[d];
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const double c = (double)loc_const;
    gb[Dp] = (gvec[2 * Dp] - 2.0 * c * gvec[2 * Dp + 1] + (double)N * c * c) - sh[0];
  }
}

int glm_recenter(GlmModel &g, const float *theta, int64_t C, cudaStream_t st) {
  dim3 gp(g.Dp / 32, kCenterSlices), bp(32, 8);
  glm_center_partial_kernel<<<gp, bp, 0, st>>>(theta, g.tf, C, g.Dtot, g.beta_off, g.D, g.Dp, g.center_part);
  glm_center_final_kernel<<<(g.Dp + 127) / 128, 128, 0, st>>>(g.center_part, g.Dp, C, g.beta0);
  if (g.form == kFormGram) {
    gram_center_kernel<<<(g.Dp + 7) / 8, 256, 0, st>>>(g.G64, g.gvec, g.beta0, g.Dp, g.loc_const, g.gb, g.gterm);
    gram_q_kernel<<<1, 256, 0, st>>>(g.gvec, g.gterm, g.Dp, g.N, g.loc_const, g.gb);
    g_launches += 4;
    B2M_CHECK_CUDA(cudaGetLastError());
    return 0;
  }
  cudaMemsetAsync(g.y0max_bits, 0, sizeof(unsigned), st);
  glm_y0_kernel<<<(g.Np + 7) / 8, 256, sizeof(float) * g.Dp, st>>>(g.X, g.y, g.beta0, g.N, g.Np, g.Dp, g.loc_const, g.y0,
                                                                   g.y0max_bits, g.lik == kLikLogit);
  g_launches += 3;
  B2M_CHECK_CUDA(cudaGetLastError());
  return 0;
}

// ---------------------------------------------------------------- pack: theta -> B = beta - beta0 (+ tf32 split), 1/sigma^2
// `idx` (optional) lists the chains of a compacted batch: row c of the batch is chain idx[c] of `theta`.
__global__ void glm_pack_kernel(const float *__restrict__ theta, const float *__restrict__ beta0,
                                const int *__restrict__ idx, int64_t C, int64_t Cp,
                                int Dtot, int beta_off, int D, int Dp, int sigma_param, float sigma_const, float *B,
                                float *Bh, float *Bl, float *inv_var) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Cp * Dp) return;
  const int64_t row = i / Dp;
  const int d = int(i % Dp);
  const int64_t c = (row < C && idx) ? idx[row] : row;
  const float v = (row < C && d < D) ? __fsub_rn(theta[c * Dtot + beta_off + d], beta0[d]) : 0.f;
  B[i] = v;
  if (Bh) {
    float hi, lo;
    split_tf32(v, hi, lo);
    Bh[i] = hi; Bl[i] = lo;
  }
  if (d == 0) {
    const float s = (row < C && sigma_param >= 0) ? theta[c * Dtot + sigma_param] : sigma_const;
    inv_var[row] = 1.0f / (s * s);
  }
}

// fp16 encoding of the A operand of K5, one warp per batch row (body: pack16_row, glm_rows.cuh)
__global__ void __launch_bounds__(128) glm_pack16_kernel(PackP P, const float *__restrict__ theta,
                                                         const int *__restrict__ idx, int64_t C, int64_t Cp) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= Cp) return;
  const int64_t c = (row < C && idx) ? idx[row] : row;
  pack16_row(P, row < C ? theta + c * P.Dtot : nullptr, row, lane);
}

// models with constraint transforms on the fp32 / tf32 paths: thc[row] = T(theta[chain of row])
__global__ void glm_constrain_kernel(const float *__restrict__ theta, const int *__restrict__ idx, const int *__restrict__ tf,
                                     int64_t C, int Dtot, float *__restrict__ thc) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= C * Dtot) return;
  const int64_t row = i / Dtot;
  const int d = int(i % Dtot);
  const int64_t c = idx ? idx[row] : row;
  thc[i] = tf_constrain(tf[d], theta[c * Dtot + d]);
}

PackP make_pack(const GlmModel &g) {
  PackP P{};
  P.beta0 = g.beta0; P.tf = g.tf; P.thc = g.thc;
  P.Dtot = g.Dtot; P.beta_off = g.beta_off; P.D = g.D; P.Dp = g.Dp; P.sigma_param = g.sigma_param;
  P.sigma_const = g.sigma_const; P.weight = g.weight;
  P.inv_col_scale = g.inv_col_scale; P.y0max_bits = g.y0max_bits; P.x_rownorm_max = g.x_rownorm_max;
  P.logit = g.lik == kLikLogit ? 1 : 0;
  P.Bh = g.B16h; P.Bl = g.B16l;
  P.inv_var = g.inv_var; P.a_unscale = g.a_unscale; P.r_scale = g.r_scale; P.r_unscale = g.r_unscale;
  if (g.form == kFormGram) { P.y0max_bits = nullptr; P.r_scale = nullptr; P.r_unscale = nullptr; }   // there is no R
  P.n_peers = 0;
  return P;
}

// ---------------------------------------------------------------- SIMT contractions (fp32, 64x64x16 tiles)
// C[m, n] = sum_k A[m, k] * Bm[n, k]; both operands K-major; all dimensions padded to the tile.
constexpr int TM = 64, TN = 64, TK = 16;

// RESID && LOGIT: the Bernoulli-logit epilogue; y = labels, eta0 = c + X beta0 (GlmModel::y0)
// STATS: the log-likelihood statistics epilogue of b2m_loglik_stats (Normal, or Bernoulli-logit with LOGIT): per
// observation and 32 draw rows, (max, sum exp(ll - max), mean, M2) into part [Cp / 32, ldc]; nothing else is written
template <bool RESID, bool LOGIT = false, bool STATS = false>
__global__ void __launch_bounds__(256) simt_gemm_kernel(const float *__restrict__ A, const float *__restrict__ Bm,
                                                        int K, int lda, int ldb, float *__restrict__ Cout, int ldc,
                                                        const float *__restrict__ y, const float *__restrict__ inv_var,
                                                        float *__restrict__ ss_part, int64_t Cp, int N_valid,
                                                        float loc_const, float weight,
                                                        const float *__restrict__ eta0 = nullptr,
                                                        float4 *__restrict__ part = nullptr, int64_t rows_valid = 0) {
  __shared__ float sA[TK][TM + 4], sB[TK][TN + 4];
  const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
  const int m0 = blockIdx.y * TM, n0 = blockIdx.x * TN;
  float acc[4][4] = {};
  const int lr = tid / 4, lc = (tid % 4) * 4;  // each thread loads one float4 of A and one of Bm per k-step
  for (int k0 = 0; k0 < K; k0 += TK) {
    const float4 a = *reinterpret_cast<const float4 *>(A + (int64_t)(m0 + lr) * lda + k0 + lc);
    const float4 b = *reinterpret_cast<const float4 *>(Bm + (int64_t)(n0 + lr) * ldb + k0 + lc);
    sA[lc + 0][lr] = a.x; sA[lc + 1][lr] = a.y; sA[lc + 2][lr] = a.z; sA[lc + 3][lr] = a.w;
    sB[lc + 0][lr] = b.x; sB[lc + 1][lr] = b.y; sB[lc + 2][lr] = b.z; sB[lc + 3][lr] = b.w;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < TK; ++k) {
      float av[4], bv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { av[i] = sA[k][ty * 4 + i]; bv[i] = sB[k][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
  if constexpr (STATS) {
    // ll per element into a [64 rows][64 columns] tile, then 128 threads reduce one column over 32 rows each, with the
    // arithmetic of the tensor-core statistics epilogue (glm_tc.cu) in the same order
    __shared__ float sl[TM][TN + 1];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int m = m0 + ty * 4 + i;
      const float iv = LOGIT ? 1.0f : inv_var[m];
      const float lbase = LOGIT ? 0.f : 0.5f * logf(iv) - kHalfLog2Pi;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int n = n0 + tx * 4 + j;
        float ll;
        if (LOGIT) {
          float dt;
          bernoulli_logit(y[n] != 0.f, eta0[n] + acc[i][j], ll, dt);
        } else {
          const float z = ((n < N_valid) ? y[n] : 0.f) - acc[i][j];
          ll = lbase - 0.5f * (iv * (z * z));
        }
        sl[ty * 4 + i][tx * 4 + j] = ll * weight;
      }
    }
    __syncthreads();
    if (tid < 2 * TN) {
      const int col = tid % TN, rg = tid / TN, n = n0 + col;
      const int64_t row0 = m0 + rg * 32, left = rows_valid - row0;
      const int nv = left >= 32 ? 32 : (left > 0 ? (int)left : 0);
      if (nv > 0 && n < N_valid) {
        float mx = -INFINITY, s = 0.f;
        for (int r = 0; r < nv; ++r) {
          const float v = sl[rg * 32 + r][col];
          mx = fmaxf(mx, v);
          s += v;
        }
        const float mean = s / (float)nv;
        float se = 0.f, m2 = 0.f;
        for (int r = 0; r < nv; ++r) {
          const float v = sl[rg * 32 + r][col];
          se += mx == -INFINITY ? 0.f : expf(v - mx);
          const float d = v - mean;
          m2 = fmaf(d, d, m2);
        }
        part[(row0 >> 5) * ldc + n] = make_float4(mx, se, mean, m2);
      }
    }
    return;
  }
  if (RESID) {
    // epilogue: z = y - c - M ; R = w z / sigma^2 ; per-row partial sum of z^2 over this column tile
    // logit:    eta = eta0 + M ; R = w (y - sigmoid(eta)) ; partial sum of y eta - softplus(eta) (padding adds 0)
    __shared__ float red[TM][17];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int m = m0 + ty * 4 + i;
      const float iv = LOGIT ? weight : inv_var[m] * weight;
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int n = n0 + tx * 4 + j;
        if (LOGIT) {
          float lp, dt;
          bernoulli_logit(y[n] != 0.f, eta0[n] + acc[i][j], lp, dt);
          s += lp;
          acc[i][j] = dt * iv;
        } else {
          const float z = (n < N_valid) ? (y[n] - loc_const) - acc[i][j] : 0.f;
          s = fmaf(z, z, s);
          acc[i][j] = z * iv;
        }
      }
      *reinterpret_cast<float4 *>(Cout + (int64_t)m * ldc + n0 + tx * 4) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
      red[ty * 4 + i][tx] = s;
    }
    __syncthreads();
    if (tid < TM) {
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < 16; ++j) s += red[tid][j];
      ss_part[(int64_t)blockIdx.x * Cp + m0 + tid] = s;
    }
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i)
      *reinterpret_cast<float4 *>(Cout + (int64_t)(m0 + ty * 4 + i) * ldc + n0 + tx * 4) =
          make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
  }
}

int simt_gemm_resid(GlmModel &g, int64_t Cp, cudaStream_t st) {
  dim3 grid(g.Np / TN, (unsigned)(Cp / TM));
  if (g.lik == kLikLogit)
    simt_gemm_kernel<true, true><<<grid, 256, 0, st>>>(g.B, g.X, g.Dp, g.Dp, g.Dp, g.R, g.Np, g.y, g.inv_var, g.ss_part,
                                                       Cp, g.N, 0.f, g.weight, g.y0);
  else
    simt_gemm_kernel<true><<<grid, 256, 0, st>>>(g.B, g.X, g.Dp, g.Dp, g.Dp, g.R, g.Np, g.y0, g.inv_var, g.ss_part, Cp,
                                                  g.N, 0.f, g.weight);
  ++g_launches;
  B2M_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int simt_gemm_stats(GlmModel &g, int64_t Cp, int64_t rows_valid, float4 *part, cudaStream_t st) {
  dim3 grid(g.Np / TN, (unsigned)(Cp / TM));
  if (g.lik == kLikLogit)
    simt_gemm_kernel<false, true, true><<<grid, 256, 0, st>>>(g.B, g.X, g.Dp, g.Dp, g.Dp, nullptr, g.Np, g.y, g.inv_var,
                                                              nullptr, Cp, g.N, 0.f, g.weight, g.y0, part, rows_valid);
  else
    simt_gemm_kernel<false, false, true><<<grid, 256, 0, st>>>(g.B, g.X, g.Dp, g.Dp, g.Dp, nullptr, g.Np, g.y0, g.inv_var,
                                                               nullptr, Cp, g.N, 0.f, g.weight, nullptr, part, rows_valid);
  ++g_launches;
  B2M_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int simt_gemm_grad(GlmModel &g, int64_t Cp, cudaStream_t st) {
  dim3 grid(g.Dp / TN, (unsigned)(Cp / TM));
  simt_gemm_kernel<false><<<grid, 256, 0, st>>>(g.R, g.XT, g.Np, g.Np, g.Np, g.G, g.Dp, nullptr, nullptr, nullptr, Cp,
                                                 0, 0.f, 0.f);
  ++g_launches;
  B2M_CHECK_CUDA(cudaGetLastError());
  return 0;
}

// ---------------------------------------------------------------- observation sharding: reduce + all-reduce
// red[c, d] = sum over split-K partials of G ; red[Cp*Dp + c] = sum over column tiles of ss_part.  Fixed order.
__global__ void __launch_bounds__(256) glm_reduce_kernel(const float *__restrict__ G, int g_splits,
                                                         const float *__restrict__ ss_part, int n_tiles, int64_t Cp,
                                                         int Dp, const float *__restrict__ r_unscale,
                                                         const float *__restrict__ inv_col_scale, float *__restrict__ red) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nG = Cp * Dp;
  if (i < nG) {
    float v = 0.f;
    for (int s = 0; s < g_splits; ++s) v += G[(int64_t)s * nG + i];
    if (r_unscale) v *= r_unscale[i / Dp] * inv_col_scale[i % Dp];   // fp16 encoding: the ranks' scales differ
    red[i] = v;
  } else if (i < nG + Cp) {
    const int64_t c = i - nG;
    float v = 0.f;
    for (int t = 0; t < n_tiles; ++t) v += ss_part[(int64_t)t * Cp + c];
    red[i] = v;
  }
}

int glm_set_comm(GlmModel &g, Comm *c, cudaStream_t st) {
  B2M_REQUIRE(!c || g.lik == kLikNormal,
              "observation sharding is defined for the Normal likelihood of the GLM class only (use chain sharding)");
  if (c)
    if (int rc = glm_use_streaming(g, "observation sharding")) return rc;
  g.comm = c;
  g.N_total = g.N;
  if (!c) return 0;
  if (g.use_tc == 2) {
    // The fp16 encoding scales every column of X by a power of two derived from the column maximum.  Ranks of an
    // observation-sharded model must use the SAME scales: with sliced state the owner of a chain packs its position
    // row (delta / col_scale) once for every rank's contraction.  Column maxima -> maximum over ranks -> re-split.
    if (int rc = comm_allreduce_f32_max(c, g.colmax, g.Dp, st)) return rc;
    col_scale_kernel<<<(g.Dp + 127) / 128, 128, 0, st>>>(reinterpret_cast<const unsigned *>(g.colmax), g.Dp, g.col_scale,
                                                         g.inv_col_scale, nullptr);
    const size_t nd = (size_t)g.Np * g.Dp;
    split_f16_kernel<<<(unsigned)((nd + 255) / 256), 256, 0, st>>>(g.X, g.Np, g.Dp, g.col_scale, g.X16h, g.X16l, g.XT16h, g.XT16l);
    g_launches += 2;
    B2M_CHECK_CUDA(cudaGetLastError());
  }
  int64_t *d = nullptr, h = g.N;
  B2M_CHECK_CUDA(cudaMalloc(&d, sizeof(int64_t)));
  B2M_CHECK_CUDA(cudaMemcpyAsync(d, &h, sizeof(h), cudaMemcpyHostToDevice, st));
  int rc = comm_allreduce_i64(c, d, 1, st);
  if (!rc) {
    cudaMemcpyAsync(&h, d, sizeof(h), cudaMemcpyDeviceToHost, st);
    cudaStreamSynchronize(st);
    g.N_total = h;
  }
  cudaFree(d);
  return rc;
}

// ---------------------------------------------------------------- finish: assemble log p and the full gradient
// One warp per chain (body: finish_row, glm_rows.cuh).  Rows [row_base, row_end) of the batch.
template <bool LIN>
__global__ void __launch_bounds__(128) glm_finish_kernel(KModel prior, FinishP F, const float *__restrict__ theta,
                                                          int64_t row_base, int64_t row_end, float *__restrict__ logp,
                                                          float *__restrict__ grad, const int *__restrict__ idx) {
  extern __shared__ __align__(16) unsigned char smem[];
  SModel sm;
  sm.n_terms = 0;
  if (F.has_prior) model_to_smem(prior, smem, sm);
  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  const int64_t c = row_base + (int64_t)blockIdx.x * (blockDim.x / 32) + warp;
  if (c >= row_end) return;
  const int64_t src = idx ? idx[c] : c;       // chain served by row c of a compacted batch
  finish_row<LIN>(F, sm, theta + src * F.Dtot, c, c, logp + src, grad ? grad + src * F.Dtot : nullptr, lane);
}

FinishP make_finish(const GlmModel &g, int64_t Cp, bool with_grad) {
  FinishP F{};
  F.has_prior = g.has_prior ? 1 : 0;
  F.Dtot = g.Dtot; F.beta_off = g.beta_off; F.D = g.D; F.Dp = g.Dp; F.sigma_param = g.sigma_param;
  F.sigma_const = g.sigma_const; F.weight = g.weight; F.N = (int)g.N_total;
  F.logit = g.lik == kLikLogit ? 1 : 0;
  F.n_tiles = g.use_tc ? g.Np / 128 : g.Np / TN;   // tcgen05: 256-wide tiles, two column halves each
  F.ss_part = g.ss_part; F.G = g.G; F.g_splits = with_grad ? (g.use_tc ? g.g_splits : 1) : 0; F.Cp = Cp;
  F.r_unscale = g.use_tc == 2 ? g.r_unscale : nullptr;
  F.inv_col_scale = g.use_tc == 2 ? g.inv_col_scale : nullptr;
  F.tf = g.tf; F.thc = g.thc;
  if (g.form == kFormGram) {   // the contraction runs for value-only calls too: log p needs delta . (G delta)
    F.gram = 1;
    F.g_splits = g.g_splits;
    F.gb = g.gb; F.beta0 = g.beta0;
    F.a_unscale = g.use_tc == 2 ? g.a_unscale : nullptr;
    F.g_unscale = g.use_tc == 2 ? g.g_unscale : nullptr;
    F.r_unscale = nullptr; F.inv_col_scale = nullptr;
  }
  return F;
}

size_t finish_smem(const GlmModel &g) { return g.has_prior ? model_smem_bytes(g.prior) : 16; }

// the finish step of the most recent contraction pair, on its own (the fused NUTS loop needs it before a recentring /
// compaction changes the row <-> chain mapping)
int glm_finish_launch(GlmModel &g, const float *theta, int64_t C, float *logp, float *grad, cudaStream_t st,
                      const int *idx, int64_t n_rows) {
  if (idx) C = n_rows;
  const int64_t Cp = C <= 128 ? 128 : (C + 255) / 256 * 256;
  const FinishP F = make_finish(g, Cp, grad != nullptr);
  (g.prior_lin ? glm_finish_kernel<true> : glm_finish_kernel<false>)<<<(unsigned)((C + 3) / 4), 128, finish_smem(g), st>>>(
      g.prior, F, theta, 0, C, logp, grad, idx);
  ++g_launches;
  B2M_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int glm_logp_grad(GlmModel &g, const float *theta, int64_t C, float *logp, float *grad, cudaStream_t st, bool recenter,
                  const int *idx, int64_t n_rows, int64_t own_base, int64_t own_count) {
  if (int rc = glm_reserve(g, C)) return rc;
  if (recenter)
    if (int rc = glm_recenter(g, theta, C, st)) return rc;
  if (idx) C = n_rows;   // compacted batch: rows 0..n_rows-1 are the chains idx[0..n_rows-1]
  const int64_t Cp = C <= 128 ? 128 : (C + 255) / 256 * 256;   // one 128-row tile, or whole 256-row CTA-pair tiles
  const int64_t tot = Cp * g.Dp;
  if (g.use_tc == 2) {
    const PackP P = make_pack(g);
    glm_pack16_kernel<<<(unsigned)((Cp + 3) / 4), 128, 0, st>>>(P, theta, idx, C, Cp);
  } else {
    const float *src = theta;
    const int *sidx = idx;
    if (g.tf) {   // the contraction sees T(theta)
      glm_constrain_kernel<<<(unsigned)((C * g.Dtot + 255) / 256), 256, 0, st>>>(theta, idx, g.tf, C, g.Dtot, g.thc);
      ++g_launches;
      src = g.thc;
      sidx = nullptr;
    }
    glm_pack_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(src, g.beta0, sidx, C, Cp, g.Dtot, g.beta_off, g.D, g.Dp,
                                                                    g.sigma_param, g.sigma_const, g.B, g.Bh, g.Bl, g.inv_var);
  }
  ++g_launches;
  if (g.use_tc && g.form == kFormGram) {
    if (int rc = tc_gemm_gram(g, Cp, st)) return rc;   // value-only too (log p needs it)
  } else if (g.use_tc) {
    if (int rc = tc_gemm_resid(g, Cp, st)) return rc;
    if (grad) if (int rc = tc_gemm_grad(g, Cp, st)) return rc;
  } else {
    if (int rc = simt_gemm_resid(g, Cp, st)) return rc;
    if (grad) if (int rc = simt_gemm_grad(g, Cp, st)) return rc;
  }
  FinishP F = make_finish(g, Cp, grad != nullptr);
  if (g.comm) {
    // observation shard: contiguous [Cp, Dp] gradient partial || [Cp] sum z^2, summed over ranks on this stream
    const int64_t n_red = Cp * g.Dp + Cp;
    glm_reduce_kernel<<<(unsigned)((n_red + 255) / 256), 256, 0, st>>>(g.G, F.g_splits, g.ss_part, F.n_tiles, Cp, g.Dp,
                                                                        F.r_unscale, F.inv_col_scale, g.red);
    ++g_launches;
    if (own_count > 0) {
      // sliced state: every rank only needs the sums of its own chains' rows -- two in-place reduce-scatters
      // (gradient block, sum-of-squares block) instead of the all-reduce
      const int nr = comm_nranks(g.comm);
      B2M_REQUIRE(!idx && Cp == C && C % nr == 0 && own_count == C / nr && own_base == own_count * comm_rank(g.comm),
                  "glm_logp_grad: sliced state needs a full batch whose rows divide evenly over the ranks");
      if (grad)
        if (int rc = comm_reducescatter_f32_inplace(g.comm, g.red, own_count * g.Dp, st)) return rc;
      if (int rc = comm_reducescatter_f32_inplace(g.comm, g.red + Cp * g.Dp, own_count, st)) return rc;
    } else {
      if (int rc = comm_allreduce_f32(g.comm, grad ? g.red : g.red + Cp * g.Dp, grad ? n_red : Cp, st)) return rc;
    }
    F.G = g.red; F.ss_part = g.red + Cp * g.Dp; F.g_splits = grad ? 1 : 0; F.n_tiles = 1;
    F.r_unscale = nullptr; F.inv_col_scale = nullptr;   // already unscaled before the sum over ranks
  }
  const int64_t row_base = (g.comm && own_count > 0) ? own_base : 0;
  const int64_t rows = (g.comm && own_count > 0) ? own_count : C;
  (g.prior_lin ? glm_finish_kernel<true> : glm_finish_kernel<false>)<<<(unsigned)((rows + 3) / 4), 128, finish_smem(g), st>>>(
      g.prior, F, theta, row_base, row_base + rows, logp, grad, idx);
  ++g_launches;
  B2M_CHECK_CUDA(cudaGetLastError());
  return 0;
}

// ---------------------------------------------------------------- pointwise log-likelihood statistics (b2m_loglik_stats)
// The centring of the samplers around beta0 = the mean of ALL draws of the call: X (theta_s - beta0) is then of the size
// of the posterior spread (same accuracy argument as for the samplers).  The next sampler or logp call recentres.
int glm_loglik_center(GlmModel &g, const float *draws, int64_t S, cudaStream_t st) {
  dim3 gp(g.Dp / 32, kCenterSlices), bp(32, 8);
  glm_center_partial_kernel<<<gp, bp, 0, st>>>(draws, nullptr, S, g.Dtot, g.beta_off, g.D, g.Dp, g.center_part);
  glm_center_final_kernel<<<(g.Dp + 127) / 128, 128, 0, st>>>(g.center_part, g.Dp, S, g.beta0);
  cudaMemsetAsync(g.y0max_bits, 0, sizeof(unsigned), st);
  glm_y0_kernel<<<(g.Np + 7) / 8, 256, sizeof(float) * g.Dp, st>>>(g.X, g.y, g.beta0, g.N, g.Np, g.Dp, g.loc_const, g.y0,
                                                                   g.y0max_bits, g.lik == kLikLogit);
  g_launches += 3;
  B2M_CHECK_CUDA(cudaGetLastError());
  return 0;
}

// One batch of `rows` draws (model coordinates: no transforms) -> partials of the X @ beta term [Cp / 32, Np].  The
// batch is packed as the samplers pack a lock-step batch (rows past `rows` are zero rows) and contracted with the
// statistics epilogue of K5.
int glm_loglik_batch(GlmModel &g, const float *draws, int64_t rows, float4 *part, cudaStream_t st) {
  if (int rc = glm_reserve(g, rows)) return rc;
  const int64_t Cp = rows <= 128 ? 128 : (rows + 255) / 256 * 256;
  if (g.use_tc == 2) {
    PackP P = make_pack(g);
    P.tf = nullptr;                           // the draws are already constrained
    P.r_scale = nullptr; P.r_unscale = nullptr;   // there is no residual operand
    glm_pack16_kernel<<<(unsigned)((Cp + 3) / 4), 128, 0, st>>>(P, draws, nullptr, rows, Cp);
  } else {
    glm_pack_kernel<<<(unsigned)((Cp * g.Dp + 255) / 256), 256, 0, st>>>(draws, g.beta0, nullptr, rows, Cp, g.Dtot, g.beta_off,
                                                                          g.D, g.Dp, g.sigma_param, g.sigma_const, g.B,
                                                                          g.Bh, g.Bl, g.inv_var);
  }
  ++g_launches;
  B2M_CHECK_CUDA(cudaGetLastError());
  if (g.use_tc) return tc_gemm_stats(g, Cp, rows, part, st);
  return simt_gemm_stats(g, Cp, rows, part, st);
}

}  // namespace b2m

// SURVEY.md 8(f) row 4: forward sampling from the six library distributions on the device (prior / posterior
// predictive draws -- the step before the sampling path).  Replaces Distribution.sample:
//   Normal       normal.py:58-77        loc + scale * N(0,1)
//   HalfNormal   halfnormal.py:65-86    |N(0,1)| * scale
//   Exponential  exponential.py:73-92   -log(U) / rate
//   Gamma        gamma.py:90-117        (the reference falls back to numpy's generator; here Marsaglia-Tsang)
//   Beta         beta.py:93-119         (numpy fallback there; here Ga / (Ga + Gb))
//   Categorical  categorical.py:95-113  inverse CDF over the normalised probabilities
//   Bernoulli    (no reference class)   U < p
// Philox4x32-10, counter = (output index, attempt, slot), key = seed: the i-th output depends only on (seed, i).
#include <math.h>

#include "common.cuh"

namespace b2m {

enum { SAMPLE_CATEGORICAL = 6 };

__device__ __forceinline__ float std_normal(uint64_t seed, uint64_t i, uint32_t attempt, uint32_t slot, float *u_extra) {
  const uint4 w = Philox::draw(seed, i, attempt, slot);
  float z0, z1;
  box_muller(w.x, w.y, z0, z1);
  if (u_extra) *u_extra = u01(w.z);
  return z0;
}

// Marsaglia & Tsang (2000) for shape >= 1; shape < 1 through Gamma(shape + 1) * U^(1 / shape)
__device__ float gamma_unit_rate(float shape, uint64_t seed, uint64_t i, uint32_t slot) {
  float boost = 1.0f;
  if (shape < 1.0f) {
    const uint4 w = Philox::draw(seed, i, 0xffffu, slot);
    boost = powf(u01(w.x), 1.0f / shape);
    shape += 1.0f;
  }
  const float d = shape - 1.0f / 3.0f, c = rsqrtf(9.0f * d);
  for (uint32_t attempt = 0; attempt < 64; ++attempt) {
    float u;
    const float x = std_normal(seed, i, attempt, slot, &u);
    const float t = 1.0f + c * x;
    if (t <= 0.f) continue;
    const float v = t * t * t;
    if (logf(u) < 0.5f * x * x + d - d * v + d * logf(v)) return boost * d * v;
  }
  return boost * d;   // 64 rejections in a row has probability < 1e-80
}

__global__ void __launch_bounds__(256) sample_kernel(int dist, float p0, float p1, const float *__restrict__ cdf, int n_cat,
                                                     uint64_t seed, int64_t n, float *__restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float r;
  switch (dist) {
    case B2M_NORMAL: r = p0 + p1 * std_normal(seed, (uint64_t)i, 0u, 0u, nullptr); break;
    case B2M_HALFNORMAL: r = fabsf(std_normal(seed, (uint64_t)i, 0u, 0u, nullptr)) * p0; break;
    case B2M_EXPONENTIAL: r = -logf(u01(Philox::draw(seed, (uint64_t)i, 0u, 0u).x)) / p0; break;
    case B2M_GAMMA: r = gamma_unit_rate(p0, seed, (uint64_t)i, 0u) / p1; break;   // p0 = alpha, p1 = rate
    case B2M_BETA: {
      const float ga = gamma_unit_rate(p0, seed, (uint64_t)i, 0u), gb = gamma_unit_rate(p1, seed, (uint64_t)i, 1u);
      r = ga / (ga + gb);
    } break;
    case B2M_BERNOULLI: r = u01(Philox::draw(seed, (uint64_t)i, 0u, 0u).x) < p0 ? 1.f : 0.f; break;   // p0 = P(1)
    case SAMPLE_CATEGORICAL: {
      const float u = u01(Philox::draw(seed, (uint64_t)i, 0u, 0u).x);
      int lo = 0, hi = n_cat - 1;   // first k with cdf[k] > u
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (cdf[mid] > u) hi = mid; else lo = mid + 1;
      }
      r = (float)lo;
    } break;
    default: r = nanf("");
  }
  out[i] = r;
}

int sample(int dist, float p0, float p1, const float *cdf, int n_cat, uint64_t seed, int64_t n, float *out, cudaStream_t st) {
  if (n == 0) return 0;
  sample_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(dist, p0, p1, cdf, n_cat, seed, n, out);
  ++g_launches;
  B2M_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace b2m

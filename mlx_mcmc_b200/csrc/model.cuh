// Device-side model: the traced term table, staged in shared memory, and the fused
// log-density + analytic gradient evaluation used by every pointwise-class kernel.
//
// Replaces: the user's log_prob + Distribution.log_prob bodies (mlx_mcmc/distributions/*.py) and
// MLX's reverse-mode pass over them (mx.grad in kernels/hmc.py:53-67, kernels/nuts.py:76-87).
// Value and gradient follow SURVEY.md 8(a2'): outside a distribution's support the term is -inf
// with zero gradient (VJP of `where`); log of a negative scale gives a NaN value with the finite
// analytic gradient.
#pragma once
#include "common.cuh"

namespace b2m {

struct DevArray {
  const float *ptr;
  int64_t rows;
  int64_t cols;
};

constexpr int kCompactTerms = 8;   // terms a "compact" model may have (their table rides in the kernel parameters)
constexpr int kCompactDim = 4;     // scalar parameters a compact model may have (theta / gradient stay in registers)

// What the host passes by value to every kernel.
struct KModel {
  const b2m_term *terms;
  const b2m_lin_entry *lin;
  const DevArray *arrays;
  int32_t n_terms, n_lin, n_arrays, D;
  int32_t stage_floats;  // total floats of the 1-D arrays staged in shared memory (0 = no staging)
  int32_t max_len;       // longest term
  // Compact models (<= kCompactTerms terms, D <= kCompactDim, no affine operands -- every model of the reference's
  // examples and tests): the term table is part of the kernel parameters, i.e. lives in the constant bank, so the
  // evaluation reads term fields as instruction operands instead of re-loading them from shared memory on every
  // gradient evaluation, and theta / gradient never leave registers (no shared-memory mailbox).
  int32_t compact;
  b2m_term cterms[kCompactTerms];
  // Constraint transforms (B2M_TF_*) per scalar parameter, pointwise class (D <= 16); has_tf = any non-zero entry.
  // GLM-class models keep their table in device memory (GlmModel::tf).
  int32_t has_tf;
  uint8_t tf[16];
};

// theta = T(u) with d theta / du and the log-Jacobian terms (include/b200mcmc.h, B2M_TF_*)
struct Tf {
  float theta, jac, dlogjac, logjac;
};
__device__ __forceinline__ Tf tf_apply(int kind, float u) {
  Tf t;
  if (kind == B2M_TF_LOG) {
    t.theta = expf(u); t.jac = t.theta; t.dlogjac = 1.0f; t.logjac = u;
  } else if (kind == B2M_TF_LOGIT) {
    const float e = expf(-fabsf(u));            // in (0, 1]: no overflow on either side
    const float s = 1.0f / (1.0f + e);          // sigmoid(|u|)
    t.theta = u >= 0.f ? s : e * s;
    t.jac = e * s * s;                          // theta (1 - theta)
    t.dlogjac = u >= 0.f ? (e - 1.0f) * s : (1.0f - e) * s;   // 1 - 2 theta
    t.logjac = -fabsf(u) - 2.0f * log1pf(e);    // log theta + log(1 - theta)
  } else {
    t.theta = u; t.jac = 1.0f; t.dlogjac = 0.0f; t.logjac = 0.0f;
  }
  return t;
}
__device__ __forceinline__ float tf_constrain(int kind, float u) {
  if (kind == B2M_TF_LOG) return expf(u);
  if (kind == B2M_TF_LOGIT) { const float e = expf(-fabsf(u)), s = 1.0f / (1.0f + e); return u >= 0.f ? s : e * s; }
  return u;
}

// Per-CTA copy in shared memory.
struct SModel {
  const b2m_term *terms;
  const b2m_lin_entry *lin;
  const DevArray *arrays;  // ptr fields point at the staged shared-memory copies when staged
  int32_t n_terms, D;
};

__host__ __device__ inline size_t align16(size_t x) { return (x + 15) & ~size_t(15); }

#ifndef __CUDACC_RTC__
__host__ inline size_t model_smem_bytes(const KModel &km) {
  return align16(sizeof(b2m_term) * km.n_terms) + align16(sizeof(b2m_lin_entry) * (km.n_lin > 0 ? km.n_lin : 1)) +
         align16(sizeof(DevArray) * (km.n_arrays > 0 ? km.n_arrays : 1)) + align16(sizeof(float) * km.stage_floats);
}
#endif

// Cooperative copy of the term table (+ float4-staged observation vectors) into shared memory.
// Returns the first free byte after the model region.
__device__ inline unsigned char *model_to_smem(const KModel &km, unsigned char *smem, SModel &sm) {
  b2m_term *terms = reinterpret_cast<b2m_term *>(smem);
  smem += align16(sizeof(b2m_term) * km.n_terms);
  b2m_lin_entry *lin = reinterpret_cast<b2m_lin_entry *>(smem);
  smem += align16(sizeof(b2m_lin_entry) * (km.n_lin > 0 ? km.n_lin : 1));
  DevArray *arrays = reinterpret_cast<DevArray *>(smem);
  smem += align16(sizeof(DevArray) * (km.n_arrays > 0 ? km.n_arrays : 1));
  float *stage = reinterpret_cast<float *>(smem);
  smem += align16(sizeof(float) * km.stage_floats);

  const int tid = threadIdx.x, nt = blockDim.x;
  {
    const uint32_t *src = reinterpret_cast<const uint32_t *>(km.terms);
    uint32_t *dst = reinterpret_cast<uint32_t *>(terms);
    for (int i = tid; i < int(sizeof(b2m_term) / 4) * km.n_terms; i += nt) dst[i] = src[i];
    const uint32_t *ls = reinterpret_cast<const uint32_t *>(km.lin);
    uint32_t *ld = reinterpret_cast<uint32_t *>(lin);
    for (int i = tid; i < int(sizeof(b2m_lin_entry) / 4) * km.n_lin; i += nt) ld[i] = ls[i];
  }
  if (tid == 0) {
    int off = 0;  // in floats, each array padded to a multiple of 4 so float4 copies stay aligned
    for (int a = 0; a < km.n_arrays; ++a) {
      DevArray d = km.arrays[a];
      if (km.stage_floats > 0 && d.cols == 1) {
        arrays[a].ptr = stage + off;
        off += int((d.rows + 3) & ~int64_t(3));
      } else {
        arrays[a].ptr = d.ptr;
      }
      arrays[a].rows = d.rows;
      arrays[a].cols = d.cols;
    }
  }
  __syncthreads();
  if (km.stage_floats > 0) {
    for (int a = 0; a < km.n_arrays; ++a) {
      DevArray d = km.arrays[a];
      if (d.cols != 1) continue;
      float *dst = const_cast<float *>(arrays[a].ptr);
      const int n4 = int(d.rows >> 2);
      if ((reinterpret_cast<uintptr_t>(d.ptr) & 15) == 0) {
        const float4 *s4 = reinterpret_cast<const float4 *>(d.ptr);
        float4 *d4 = reinterpret_cast<float4 *>(dst);
        for (int i = tid; i < n4; i += nt) d4[i] = __ldg(s4 + i);  // coalesced 16-byte loads
        for (int i = (n4 << 2) + tid; i < d.rows; i += nt) dst[i] = __ldg(d.ptr + i);
      } else {
        for (int i = tid; i < d.rows; i += nt) dst[i] = __ldg(d.ptr + i);
      }
    }
  }
  __syncthreads();
  sm.terms = terms;
  sm.lin = lin;
  sm.arrays = arrays;
  sm.n_terms = km.n_terms;
  sm.D = km.D;
  return smem;
}

// ---------------------------------------------------------------- operands
// `th` / `gr` are this lane's private columns of the shared-memory mailboxes: element d lives at
// [d * TS], TS = blockDim.x, so consecutive threads hit consecutive banks.
__device__ __forceinline__ bool op_varies(const b2m_operand &o) {
  return o.kind == B2M_OP_DATA || o.kind == B2M_OP_PARAMVEC || o.kind == B2M_OP_LIN;
}

__device__ __forceinline__ float op_fetch(const b2m_operand &o, int n, const float *th, int TS, const SModel &sm) {
  switch (o.kind) {
    case B2M_OP_PARAM: return th[o.a * TS];
    case B2M_OP_DATA: return sm.arrays[o.a].ptr[n];
    case B2M_OP_PARAMVEC: return th[(o.a + n) * TS];
    case B2M_OP_LIN: {
      float v = o.c;
      for (int e = o.a; e < o.a + o.b; ++e) {
        b2m_lin_entry le = sm.lin[e];
        float t = le.coef;
        if (le.array >= 0) t *= sm.arrays[le.array].ptr[n];
        if (le.param >= 0) t *= th[le.param * TS];
        v += t;
      }
      return v;
    }
    default: return o.c;
  }
}

__device__ __forceinline__ void op_scatter(const b2m_operand &o, int n, float adj, float *gr, int TS,
                                           const SModel &sm) {
  switch (o.kind) {
    case B2M_OP_PARAM: gr[o.a * TS] += adj; break;
    case B2M_OP_PARAMVEC: gr[(o.a + n) * TS] += adj; break;
    case B2M_OP_LIN:
      for (int e = o.a; e < o.a + o.b; ++e) {
        b2m_lin_entry le = sm.lin[e];
        if (le.param < 0) continue;
        float t = le.coef;
        if (le.array >= 0) t *= sm.arrays[le.array].ptr[n];
        gr[le.param * TS] += adj * t;
      }
      break;
    default: break;
  }
}

// ---------------------------------------------------------------- densities
constexpr float kHalfLog2Pi = 0.91893853320467274178f;
constexpr float kLog2 = 0.69314718055994530942f;

struct Elem {
  float lp, dx, d0, d1;
};

// Bernoulli with logit t and label y (one = y is 1): lp = y t - softplus(t), dt = d lp / dt = y - sigmoid(t), both from one
// e = exp(-|t|) in (0, 1].  y t - max(t, 0) is 0 when the label agrees with the sign of t and -|t| otherwise, and
// y - sigmoid(t) is +-sigmoid(-|t|) or +-sigmoid(|t|): no cancellation and no overflow at any |t| (inf included).
// Shared by the pointwise density below and the residual epilogues of the GLM contractions (glm.cu, glm_tc.cu).
__device__ __forceinline__ void bernoulli_logit(bool one, float t, float &lp, float &dt) {
  const float e = expf(-fabsf(t));
  const float r = 1.0f / (1.0f + e);   // sigmoid(|t|)
  const bool match = one == (t >= 0.f);
  lp = (match ? 0.f : -fabsf(t)) - log1pf(e);
  const float m = match ? e * r : r;
  dt = one ? m : -m;
}

template <bool GRAD>
__device__ __forceinline__ Elem dist_eval(int dist, float x, float p0, float p1, float k0, float k1, float k2) {
  Elem e;
  e.lp = 0.f; e.dx = 0.f; e.d0 = 0.f; e.d1 = 0.f;
  const float ninf = -INFINITY;
  switch (dist) {
    case B2M_NORMAL: {  // normal.py:49-56
      float z = x - p0, var = p1 * p1;
      e.lp = (-kHalfLog2Pi - logf(p1)) - (0.5f * (z * z)) / var;
      if (GRAD) {
        float t = z / var;
        e.dx = -t; e.d0 = t; e.d1 = z * t / p1 - 1.0f / p1;
      }
    } break;
    case B2M_HALFNORMAL: {  // halfnormal.py:55-63
      if (x >= 0.f) {
        float var = p0 * p0;
        e.lp = ((kLog2 + -kHalfLog2Pi) - logf(p0)) - (0.5f * (x * x)) / var;
        if (GRAD) {
          float t = x / var;
          e.dx = -t; e.d0 = x * t / p0 - 1.0f / p0;
        }
      } else {
        e.lp = ninf;
      }
    } break;
    case B2M_EXPONENTIAL: {  // exponential.py:61-71
      if (x >= 0.f) {
        e.lp = logf(p0) - p0 * x;
        if (GRAD) { e.dx = -p0; e.d0 = 1.0f / p0 - x; }
      } else {
        e.lp = ninf;
      }
    } break;
    case B2M_GAMMA: {  // gamma.py:53-88 ; p0 = rate, k0 = alpha, k1 = lgamma(alpha)
      if (x > 0.f) {
        e.lp = (k0 * logf(p0) - k1) + (k0 - 1.0f) * logf(x) - p0 * x;
        if (GRAD) { e.dx = (k0 - 1.0f) / x - p0; e.d0 = k0 / p0 - x; }
      } else {
        e.lp = ninf;
      }
    } break;
    case B2M_BETA: {  // beta.py:53-91 ; k0 = a, k1 = b, k2 = log B(a, b)
      if (x > 0.f && x < 1.f) {
        e.lp = (k0 - 1.0f) * logf(x) + (k1 - 1.0f) * logf(1.0f - x) - k2;
        if (GRAD) e.dx = (k0 - 1.0f) / x - (k1 - 1.0f) / (1.0f - x);
      } else {
        e.lp = ninf;
      }
    } break;
    case B2M_BERNOULLI: {  // x = label, p0 = logit
      if (x == 0.f || x == 1.f) {
        float lp, dt;
        bernoulli_logit(x == 1.f, p0, lp, dt);
        e.lp = lp;
        if (GRAD) e.d0 = dt;
      } else {
        e.lp = ninf;
      }
    } break;
    default: e.lp = k0; break;  // B2M_CONSTANT
  }
  return e;
}

// ---------------------------------------------------------------- fused value + gradient
// One chain is served by G lanes (G in {1,2,..,32}, a power of two, lanes contiguous in the warp).
// Each lane walks elements n = lane, lane+G, ... of every term; the G partial sums are combined
// with xor shuffles so every lane ends with the identical total.
//   th : this lane's theta mailbox column (read)      -- all G lanes hold the same values
//   gr : this lane's gradient mailbox column (written) -- after the call every lane holds d logp/d theta
template <bool GRAD>
__device__ inline float eval_model(const SModel &sm, const float *th, float *gr, int TS, int lane, int G,
                                   unsigned gmask) {
  float total = 0.f;
  if (GRAD)
    for (int d = 0; d < sm.D; ++d) gr[d * TS] = 0.f;

  for (int t = 0; t < sm.n_terms; ++t) {
    const b2m_term &T = sm.terms[t];
    const b2m_operand ox = T.x, o0 = T.p0, o1 = T.p1;
    const int dist = T.dist, len = T.length;
    const float k0 = T.k0, k1 = T.k1, k2 = T.k2, w = T.weight;
    float acc = 0.f, ax = 0.f, a0 = 0.f, a1 = 0.f;

    const bool params_fixed = !op_varies(o0) && !op_varies(o1);
    if (params_fixed && ox.kind == B2M_OP_DATA && dist == B2M_NORMAL) {
      // Hot pattern (C1 likelihood): Normal(mu, sigma) over an observation vector.  Four independent
      // accumulators per statistic: breaks the FADD dependency chain and shortens each rounding chain.
      const float mu = op_fetch(o0, 0, th, TS, sm), sg = op_fetch(o1, 0, th, TS, sm);
      const float inv_var = 1.0f / (sg * sg), base = -kHalfLog2Pi - logf(sg);
      const float *y = sm.arrays[ox.a].ptr;
      float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
      int n = lane;
      if (G == 1 && (reinterpret_cast<uintptr_t>(y) & 15) == 0) {
        const float4 *y4 = reinterpret_cast<const float4 *>(y);
        for (; n + 3 < len; n += 4) {  // one 16-byte broadcast load per four observations
          const float4 v = y4[n >> 2];
          const float z0 = v.x - mu, z1 = v.y - mu, z2 = v.z - mu, z3 = v.w - mu;
          s1[0] += z0; s1[1] += z1; s1[2] += z2; s1[3] += z3;
          s2[0] = fmaf(z0, z0, s2[0]); s2[1] = fmaf(z1, z1, s2[1]);
          s2[2] = fmaf(z2, z2, s2[2]); s2[3] = fmaf(z3, z3, s2[3]);
        }
      } else {
        for (; n + 3 * G < len; n += 4 * G) {
          const float z0 = y[n] - mu, z1 = y[n + G] - mu, z2 = y[n + 2 * G] - mu, z3 = y[n + 3 * G] - mu;
          s1[0] += z0; s1[1] += z1; s1[2] += z2; s1[3] += z3;
          s2[0] = fmaf(z0, z0, s2[0]); s2[1] = fmaf(z1, z1, s2[1]);
          s2[2] = fmaf(z2, z2, s2[2]); s2[3] = fmaf(z3, z3, s2[3]);
        }
      }
      for (; n < len; n += G) {
        const float z = y[n] - mu;
        s1[0] += z;
        s2[0] = fmaf(z, z, s2[0]);
      }
      const float t1 = (s1[0] + s1[1]) + (s1[2] + s1[3]), t2 = (s2[0] + s2[1]) + (s2[2] + s2[3]);
      const float cnt = (float)((len - lane + G - 1) / G);
      acc = cnt * base - 0.5f * t2 * inv_var;
      a0 = t1 * inv_var;
      a1 = (t2 * inv_var - cnt) / sg;
    } else if (params_fixed && ox.kind == B2M_OP_DATA && dist == B2M_EXPONENTIAL) {
      // Hot pattern (C2 likelihood): Exponential(rate) over an observation vector.
      const float rate = op_fetch(o0, 0, th, TS, sm);
      const float lr = logf(rate), ir = 1.0f / rate;
      const float *y = sm.arrays[ox.a].ptr;
      float s1[4] = {0.f, 0.f, 0.f, 0.f};
      float lo = INFINITY;  // min over the data: a negative (or NaN) datum is outside the support
      int n = lane;
      if (G == 1 && (reinterpret_cast<uintptr_t>(y) & 15) == 0) {
        const float4 *y4 = reinterpret_cast<const float4 *>(y);
        for (; n + 3 < len; n += 4) {
          const float4 v = y4[n >> 2];
          s1[0] += v.x; s1[1] += v.y; s1[2] += v.z; s1[3] += v.w;
          lo = fminf(fminf(lo, fminf(v.x, v.y)), fminf(v.z, v.w));
        }
      } else {
        for (; n + 3 * G < len; n += 4 * G) {
          const float v0 = y[n], v1 = y[n + G], v2 = y[n + 2 * G], v3 = y[n + 3 * G];
          s1[0] += v0; s1[1] += v1; s1[2] += v2; s1[3] += v3;
          lo = fminf(fminf(lo, fminf(v0, v1)), fminf(v2, v3));
        }
      }
      for (; n < len; n += G) {
        const float v = y[n];
        s1[0] += v;
        lo = fminf(lo, v);
      }
      const float t1 = (s1[0] + s1[1]) + (s1[2] + s1[3]);
      const float cnt = (float)((len - lane + G - 1) / G);
      const bool bad = !(lo >= 0.f) || !(t1 == t1);
      if (!bad) {
        acc = cnt * lr - rate * t1;
        a0 = cnt * ir - t1;
      } else {  // some datum outside the support: -inf value, masked per-element gradient (rare path)
        acc = -INFINITY;
        a0 = 0.f;
        for (int m = lane; m < len; m += G) {
          const float v = y[m];
          if (v >= 0.f) a0 += ir - v;
        }
      }
    } else {
      for (int n = lane; n < len; n += G) {
        const float x = op_fetch(ox, n, th, TS, sm);
        const float p0 = op_fetch(o0, n, th, TS, sm);
        const float p1 = op_fetch(o1, n, th, TS, sm);
        Elem e = dist_eval<GRAD>(dist, x, p0, p1, k0, k1, k2);
        acc += e.lp;
        if (GRAD) {
          if (ox.kind == B2M_OP_PARAM) ax += e.dx; else op_scatter(ox, n, w * e.dx, gr, TS, sm);
          if (o0.kind == B2M_OP_PARAM) a0 += e.d0; else op_scatter(o0, n, w * e.d0, gr, TS, sm);
          if (o1.kind == B2M_OP_PARAM) a1 += e.d1; else op_scatter(o1, n, w * e.d1, gr, TS, sm);
        }
      }
    }
    total += w * acc;
    if (GRAD) {
      if (ox.kind == B2M_OP_PARAM) gr[ox.a * TS] += w * ax;
      if (o0.kind == B2M_OP_PARAM) gr[o0.a * TS] += w * a0;
      if (o1.kind == B2M_OP_PARAM) gr[o1.a * TS] += w * a1;
    }
  }

  // combine the G lanes of the chain; gmask names exactly those lanes, so chains sharing a warp may
  // diverge from each other (NUTS tree depth) without breaking the shuffles
  for (int o = G >> 1; o > 0; o >>= 1) total += __shfl_xor_sync(gmask, total, o);
  if (GRAD && G > 1) {
    for (int d = 0; d < sm.D; ++d) {
      float v = gr[d * TS];
      for (int o = G >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(gmask, v, o);
      gr[d * TS] = v;
    }
  }
  return total;
}

// ---------------------------------------------------------------- compact models: registers + constant bank
template <int DMAX>
__device__ __forceinline__ float reg_get(const float (&q)[DMAX], int i) {
  float v = q[0];
#pragma unroll
  for (int d = 1; d < DMAX; ++d) v = (i == d) ? q[d] : v;
  return v;
}
template <int DMAX>
__device__ __forceinline__ void reg_add(float (&g)[DMAX], int i, float v) {
#pragma unroll
  for (int d = 0; d < DMAX; ++d)
    if (i == d) g[d] += v;
}

template <int DMAX>
__device__ __forceinline__ float op_fetch_c(const b2m_operand &o, int n, const float (&q)[DMAX], const SModel &sm) {
  switch (o.kind) {
    case B2M_OP_PARAM: return reg_get<DMAX>(q, o.a);
    case B2M_OP_DATA: return sm.arrays[o.a].ptr[n];
    case B2M_OP_PARAMVEC: return reg_get<DMAX>(q, o.a + n);
    default: return o.c;
  }
}
template <int DMAX>
__device__ __forceinline__ void op_scatter_c(const b2m_operand &o, int n, float adj, float (&g)[DMAX]) {
  if (o.kind == B2M_OP_PARAM) reg_add<DMAX>(g, o.a, adj);
  else if (o.kind == B2M_OP_PARAMVEC) reg_add<DMAX>(g, o.a + n, adj);
}

// One term of a compact / specialised model: same arithmetic, in the same order, as eval_model (so the paths agree bit
// for bit).  Generic kernels pass `km.cterms[t]` of their __grid_constant__ parameter (constant-bank operands); the
// NVRTC-specialised kernels (jit.cu, mlx_mcmc_b200/jit.py) pass a term built from literals, so that after inlining
// every switch on the distribution, every operand kind and every constant folds away.
template <bool GRAD, int DMAX>
__device__ __forceinline__ void eval_term_c(const b2m_term &T, const SModel &sm, const float (&q)[DMAX], float (&g)[DMAX],
                                            int lane, int G, float &total) {
  const int dist = T.dist, len = T.length;
  const float k0 = T.k0, k1 = T.k1, k2 = T.k2, w = T.weight;
  float acc = 0.f, ax = 0.f, a0 = 0.f, a1 = 0.f;
  const bool params_fixed = !op_varies(T.p0) && !op_varies(T.p1);
  if (params_fixed && T.x.kind == B2M_OP_DATA && dist == B2M_NORMAL) {
    const float mu = op_fetch_c<DMAX>(T.p0, 0, q, sm), sg = op_fetch_c<DMAX>(T.p1, 0, q, sm);
    const float inv_var = 1.0f / (sg * sg), base = -kHalfLog2Pi - logf(sg);
    const float *y = sm.arrays[T.x.a].ptr;
    float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
    int n = lane;
    if (G == 1 && (reinterpret_cast<uintptr_t>(y) & 15) == 0) {
      const float4 *y4 = reinterpret_cast<const float4 *>(y);
      for (; n + 3 < len; n += 4) {
        const float4 v = y4[n >> 2];
        const float z0 = v.x - mu, z1 = v.y - mu, z2 = v.z - mu, z3 = v.w - mu;
        s1[0] += z0; s1[1] += z1; s1[2] += z2; s1[3] += z3;
        s2[0] = fmaf(z0, z0, s2[0]); s2[1] = fmaf(z1, z1, s2[1]);
        s2[2] = fmaf(z2, z2, s2[2]); s2[3] = fmaf(z3, z3, s2[3]);
      }
    } else {
      for (; n + 3 * G < len; n += 4 * G) {
        const float z0 = y[n] - mu, z1 = y[n + G] - mu, z2 = y[n + 2 * G] - mu, z3 = y[n + 3 * G] - mu;
        s1[0] += z0; s1[1] += z1; s1[2] += z2; s1[3] += z3;
        s2[0] = fmaf(z0, z0, s2[0]); s2[1] = fmaf(z1, z1, s2[1]);
        s2[2] = fmaf(z2, z2, s2[2]); s2[3] = fmaf(z3, z3, s2[3]);
      }
    }
    for (; n < len; n += G) {
      const float z = y[n] - mu;
      s1[0] += z;
      s2[0] = fmaf(z, z, s2[0]);
    }
    const float t1 = (s1[0] + s1[1]) + (s1[2] + s1[3]), t2 = (s2[0] + s2[1]) + (s2[2] + s2[3]);
    const float cnt = (float)((len - lane + G - 1) / G);
    acc = cnt * base - 0.5f * t2 * inv_var;
    a0 = t1 * inv_var;
    a1 = (t2 * inv_var - cnt) / sg;
  } else if (params_fixed && T.x.kind == B2M_OP_DATA && dist == B2M_EXPONENTIAL) {
    const float rate = op_fetch_c<DMAX>(T.p0, 0, q, sm);
    const float lr = logf(rate), ir = 1.0f / rate;
    const float *y = sm.arrays[T.x.a].ptr;
    float s1[4] = {0.f, 0.f, 0.f, 0.f};
    float lo = INFINITY;
    int n = lane;
    if (G == 1 && (reinterpret_cast<uintptr_t>(y) & 15) == 0) {
      const float4 *y4 = reinterpret_cast<const float4 *>(y);
      for (; n + 3 < len; n += 4) {
        const float4 v = y4[n >> 2];
        s1[0] += v.x; s1[1] += v.y; s1[2] += v.z; s1[3] += v.w;
        lo = fminf(fminf(lo, fminf(v.x, v.y)), fminf(v.z, v.w));
      }
    } else {
      for (; n + 3 * G < len; n += 4 * G) {
        const float v0 = y[n], v1 = y[n + G], v2 = y[n + 2 * G], v3 = y[n + 3 * G];
        s1[0] += v0; s1[1] += v1; s1[2] += v2; s1[3] += v3;
        lo = fminf(fminf(lo, fminf(v0, v1)), fminf(v2, v3));
      }
    }
    for (; n < len; n += G) {
      const float v = y[n];
      s1[0] += v;
      lo = fminf(lo, v);
    }
    const float t1 = (s1[0] + s1[1]) + (s1[2] + s1[3]);
    const float cnt = (float)((len - lane + G - 1) / G);
    const bool bad = !(lo >= 0.f) || !(t1 == t1);
    if (!bad) {
      acc = cnt * lr - rate * t1;
      a0 = cnt * ir - t1;
    } else {
      acc = -INFINITY;
      a0 = 0.f;
      for (int m = lane; m < len; m += G) {
        const float v = y[m];
        if (v >= 0.f) a0 += ir - v;
      }
    }
  } else {
    for (int n = lane; n < len; n += G) {
      const float x = op_fetch_c<DMAX>(T.x, n, q, sm);
      const float p0 = op_fetch_c<DMAX>(T.p0, n, q, sm);
      const float p1 = op_fetch_c<DMAX>(T.p1, n, q, sm);
      Elem e = dist_eval<GRAD>(dist, x, p0, p1, k0, k1, k2);
      acc += e.lp;
      if (GRAD) {
        if (T.x.kind == B2M_OP_PARAM) ax += e.dx; else op_scatter_c<DMAX>(T.x, n, w * e.dx, g);
        if (T.p0.kind == B2M_OP_PARAM) a0 += e.d0; else op_scatter_c<DMAX>(T.p0, n, w * e.d0, g);
        if (T.p1.kind == B2M_OP_PARAM) a1 += e.d1; else op_scatter_c<DMAX>(T.p1, n, w * e.d1, g);
      }
    }
  }
  total += w * acc;
  if (GRAD) {
    if (T.x.kind == B2M_OP_PARAM) reg_add<DMAX>(g, T.x.a, w * ax);
    if (T.p0.kind == B2M_OP_PARAM) reg_add<DMAX>(g, T.p0.a, w * a0);
    if (T.p1.kind == B2M_OP_PARAM) reg_add<DMAX>(g, T.p1.a, w * a1);
  }
}

#ifdef B2M_JIT
// a constant of the term table whose VALUE the compiler cannot see (control flow on the integer fields still folds):
// arithmetic on it runs on the device exactly as in the generic kernels, which keeps the two bit-identical
__device__ __forceinline__ float jit_const(unsigned bits) {
  float v;
  asm("mov.b32 %0, %1;" : "=f"(v) : "r"(bits));
  return v;
}
// the generated translation unit defines B2M_JIT_TERMS(F): one F(dist, length, weight, k0, k1, k2, x.kind, x.a, x.b, x.c,
// p0.kind, p0.a, p0.b, p0.c, p1.kind, p1.a, p1.b, p1.c) per term of the traced model
#define B2M_JIT_ONE_TERM(DIST, LEN, W, K0, K1, K2, XK, XA, XB, XC, AK, AA, AB, AC, BK, BA, BB, BC)                      \
  {                                                                                                                      \
    const b2m_term T = {DIST, LEN, W, K0, K1, K2, {XK, XA, XB, XC}, {AK, AA, AB, AC}, {BK, BA, BB, BC}};                  \
    eval_term_c<GRAD, DMAX>(T, sm, q, g, lane, G, total);                                                                \
  }
#endif

template <bool GRAD, int DMAX>
__device__ __forceinline__ float eval_model_c(const KModel &km, const SModel &sm, const float (&q)[DMAX], float (&g)[DMAX],
                                              int lane, int G, unsigned gmask) {
  float total = 0.f;
  if (GRAD) {
#pragma unroll
    for (int d = 0; d < DMAX; ++d) g[d] = 0.f;
  }
#ifdef B2M_JIT
  (void)km;
  B2M_JIT_TERMS(B2M_JIT_ONE_TERM)
#else
#pragma unroll
  for (int t = 0; t < kCompactTerms; ++t) {
    if (t >= km.n_terms) break;
    eval_term_c<GRAD, DMAX>(km.cterms[t], sm, q, g, lane, G, total);
  }
#endif
  for (int o = G >> 1; o > 0; o >>= 1) total += __shfl_xor_sync(gmask, total, o);
  if (GRAD && G > 1) {
#pragma unroll
    for (int d = 0; d < DMAX; ++d) {
      float v = g[d];
      for (int o = G >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(gmask, v, o);
      g[d] = v;
    }
  }
  return total;
}

}  // namespace b2m

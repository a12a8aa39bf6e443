// Per-row device bodies of the GLM evaluation pipeline (one warp per chain row), shared by the stand-alone kernels
// of glm.cu and by the fused NUTS state kernel of glm_samplers.cu (finish of leaf t-1 + tree bookkeeping + pack of
// leaf t in one launch).  Same arithmetic, in the same order, wherever they are called from.
#pragma once
#include "glm.cuh"

namespace b2m {

// power-of-two scale that puts a maximum of `m` just below 2^14 (fp16 overflows at 65504 = 2^16 - 32)
__host__ __device__ inline float pow2_scale(float m) {
  if (!(m > 0.f) || !(m < 3.0e38f)) return 1.0f;
  int e;
  frexpf(m, &e);                 // m = f * 2^e, f in [0.5, 1)  =>  m < 2^e
  int k = 14 - e;
  if (k > 100) k = 100;
  if (k < -100) k = -100;
  return ldexpf(1.0f, k);
}

__device__ __forceinline__ void split_f16(float v, __half &hi, __half &lo) {
  hi = __float2half_rn(v);
  lo = __float2half_rn(v - __half2float(hi));
}

// ---------------------------------------------------------------- pack (fp16 encoding)
struct PackP {
  const float *beta0;
  const int *tf;          // [Dtot] transform codes or nullptr
  float *thc;             // [Cp, Dtot] constrained copy of the batch rows (written only when tf != nullptr)
  int Dtot, beta_off, D, Dp, sigma_param;
  float sigma_const, weight;
  const float *inv_col_scale;
  const unsigned *y0max_bits;
  float x_rownorm_max;
  int logit;              // GlmModel::lik == kLikLogit: |R| <= |w|, the row scale of R needs no data bound
  __half *Bh, *Bl;        // [Cp, Dp]
  float *inv_var, *a_unscale, *r_scale, *r_unscale;   // [Cp]
  // peer window (sliced observation sharding): the row is written into every rank's window instead, with the row
  // scalars as one float4 (the receiving rank derives its own r_scale from ||delta||^2: its y0 maximum is local)
  int n_peers;
  __half *peer_Bh[kMaxPeers], *peer_Bl[kMaxPeers];
  float4 *peer_meta[kMaxPeers];
};

// fp16 encoding of the A operand of K5 for batch row `row` <- parameter row `th` (nullptr: a padding row of zeros):
//   delta'_d = (beta_d - beta0_d) / col_scale_d          (X' = X col_scale, so delta' . X' = delta . X exactly)
//   row scale s_a = 2^k putting max_d |delta'_d| just below 2^14; hi / lo halves of delta' s_a
// and the row scale of the residual operand of K6 from a bound that is known before K5 runs:
//   Normal: |z_n| = |y0_n - (X delta)_n| <= max|y0| + ||delta||_2 max_n ||X_n||_2      (Cauchy-Schwarz)
//   logit:  |R_n| = |w| |y_n - sigmoid(eta_n)| <= |w|
__device__ __forceinline__ void pack16_row(const PackP &P, const float *__restrict__ th, int64_t row, int lane) {
  const bool live = th != nullptr;
  B2M_ASSERT(row >= 0 && P.Dp % 64 == 0 && P.D <= P.Dp && P.beta_off + P.D <= P.Dtot);
  const int *tf = P.tf;
  float amax = 0.f, n2 = 0.f;
  if (live) {
    if (tf) {   // the model sees T(u): keep the constrained row for finish (priors, sigma)
      float *tc = P.thc + row * P.Dtot;
      for (int d = lane; d < P.Dtot; d += 32) tc[d] = tf_constrain(tf[d], th[d]);
      __syncwarp();
      th = tc;
    }
    for (int d = lane; d < P.D; d += 32) {
      const float dl = __fsub_rn(th[P.beta_off + d], P.beta0[d]);
      amax = fmaxf(amax, fabsf(dl * P.inv_col_scale[d]));
      n2 = fmaf(dl, dl, n2);
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
    n2 += __shfl_xor_sync(0xffffffffu, n2, o);
  }
  const float sa = pow2_scale(amax);
  const float sg = (live && P.sigma_param >= 0) ? th[P.sigma_param] : P.sigma_const;
  const float iv = 1.0f / (sg * sg);
  if (P.n_peers == 0) {
    for (int d = lane; d < P.Dp; d += 32) {
      float v = 0.f;
      if (live && d < P.D) v = __fsub_rn(th[P.beta_off + d], P.beta0[d]) * P.inv_col_scale[d] * sa;
      __half hi, lo;
      split_f16(v, hi, lo);
      P.Bh[row * P.Dp + d] = hi;
      P.Bl[row * P.Dp + d] = lo;
    }
    if (lane == 0) {
      P.inv_var[row] = iv;
      P.a_unscale[row] = 1.0f / sa;
      if (P.r_scale) {   // streaming form only: the Gram form has no residual operand
        const float bound = P.logit ? fabsf(P.weight)
                                    : (__uint_as_float(*P.y0max_bits) + sqrtf(n2) * P.x_rownorm_max) * fabsf(iv * P.weight);
        const float sr = pow2_scale(bound);
        P.r_scale[row] = sr;
        P.r_unscale[row] = 1.0f / sr;
      }
    }
  } else {
    // two coefficients per lane and store: 128-byte segments per warp instruction towards every peer over NVLink
    for (int d = 2 * lane; d < P.Dp; d += 64) {
      float v0 = 0.f, v1 = 0.f;
      if (live && d < P.D) v0 = __fsub_rn(th[P.beta_off + d], P.beta0[d]) * P.inv_col_scale[d] * sa;
      if (live && d + 1 < P.D) v1 = __fsub_rn(th[P.beta_off + d + 1], P.beta0[d + 1]) * P.inv_col_scale[d + 1] * sa;
      const __half2 hi = __floats2half2_rn(v0, v1);
      const float2 hf = __half22float2(hi);
      const __half2 lo = __floats2half2_rn(v0 - hf.x, v1 - hf.y);
#pragma unroll
      for (int s = 0; s < kMaxPeers; ++s)
        if (s < P.n_peers) {
          *reinterpret_cast<__half2 *>(P.peer_Bh[s] + row * P.Dp + d) = hi;
          *reinterpret_cast<__half2 *>(P.peer_Bl[s] + row * P.Dp + d) = lo;
        }
    }
    if (lane < P.n_peers) P.peer_meta[lane][row] = make_float4(iv, 1.0f / sa, n2, 0.f);
  }
}

// ---------------------------------------------------------------- finish
struct FinishP {
  int has_prior;
  int Dtot, beta_off, D, Dp, sigma_param;
  float sigma_const, weight;
  int N;                 // observations of the whole model (all shards)
  int logit;             // GlmModel::lik == kLikLogit: the partial sums are the log-likelihood itself, no sigma
  int n_tiles;           // partial sums of z^2 (or of the Bernoulli terms) per row
  const float *ss_part;  // [n_tiles, Cp]
  const float *G;        // [g_splits, Cp, Dp]
  int g_splits;
  int64_t Cp;            // row stride of ss_part / G
  const float *r_unscale;      // [Cp] or nullptr
  const float *inv_col_scale;  // [Dp] or nullptr
  const int *tf;         // transforms or nullptr
  const float *thc;      // [Cp, Dtot] constrained rows written by pack (tf != nullptr)
  // Gram form (GlmModel::form): G holds the split-K partials of P = delta G~ instead, ss_part is unused
  int gram;
  const double *gb;          // [Dp + 1] b = X^T y0 || q = ||y0||^2 of the current centring
  const float *beta0;        // [Dp]
  const float *a_unscale;    // [Cp] 1 / row scale of the packed delta (fp16 encoding) or nullptr
  const float *g_unscale;    // [Dp] 1 / (cs_j t_j) (fp16 encoding) or nullptr
};

// Gram form, likelihood part of one row: P = sum of the split-K partials (fixed order), unscaled;
//     grad_beta = w iv (b - P),   ss = q - 2 delta.b + delta.P   (float64 across the warp, fixed order)
// with delta = theta_beta - beta0 exactly as pack computed it.  The lane <-> coefficient mapping depends on D only,
// never on whether a gradient is wanted: a value-only call gets the bit-identical ss.  Returns ss (every lane).
__device__ __forceinline__ float gram_row(const FinishP &F, const float *__restrict__ th, int64_t c, float ivw,
                                          float *__restrict__ gr, int lane) {
  const int D = F.D, Dp = F.Dp, beta_off = F.beta_off;
  const int64_t stride = F.Cp * (int64_t)Dp;
  const float *__restrict__ Gr = F.G + c * Dp;
  const float au = F.a_unscale ? F.a_unscale[c] : 1.0f;
  const int step = (D & 3) == 0 ? 4 : 1;   // four consecutive coefficients per lane: independent 16-byte loads
  double acc = 0.0;
  for (int j0 = step * lane; j0 < D; j0 += 32 * step) {
    float p[4] = {0.f, 0.f, 0.f, 0.f};
    if (step == 4) {
#pragma unroll 4
      for (int s = 0; s < F.g_splits; ++s) {
        const float4 t = *reinterpret_cast<const float4 *>(Gr + s * stride + j0);
        p[0] += t.x; p[1] += t.y; p[2] += t.z; p[3] += t.w;
      }
    } else {
#pragma unroll 4
      for (int s = 0; s < F.g_splits; ++s) p[0] += Gr[s * stride + j0];
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      if (e >= step) break;
      const int j = j0 + e;
      const float pj = F.g_unscale ? p[e] * (au * F.g_unscale[j]) : p[e];
      const double bj = F.gb[j];
      const float dl = __fsub_rn(th[beta_off + j], F.beta0[j]);
      acc += (double)dl * ((double)pj - 2.0 * bj);
      if (gr) gr[beta_off + j] = (float)(bj - (double)pj) * ivw;
    }
  }
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  return (float)(F.gb[Dp] + acc);
}

// Assemble log p and the full gradient of one chain from the contraction outputs.  `c` = row of ss_part / G (and of
// thc); `th` = the chain's parameter row as the samplers hold it (unconstrained when tf is set); logp / gr = outputs.
// Likelihood value from the partial sums (fixed summation order => deterministic), gradient of beta from G, gradient
// of sigma analytically, then the prior terms (generic densities) added on top.
__device__ __forceinline__ void finish_row(const FinishP &F, const SModel &sm, const float *__restrict__ th, int64_t c,
                                           int64_t c_batch, float *__restrict__ logp_out, float *__restrict__ gr, int lane) {
  B2M_ASSERT(c >= 0 && c < F.Cp && F.g_splits >= 0 && F.n_tiles >= 1);
  const float *thu = th;                         // unconstrained row (chain rule below)
  if (F.tf) th = F.thc + c_batch * F.Dtot;       // the model's view (c_batch = row of the packed batch)
  const int Dtot = F.Dtot, D = F.D, Dp = F.Dp, beta_off = F.beta_off, sigma_param = F.sigma_param;
  const int64_t Cp = F.Cp;
  const float *__restrict__ G = F.G;
  const float sg = sigma_param >= 0 ? th[sigma_param] : F.sigma_const;
  const float iv = 1.0f / (sg * sg);
  const float weight = F.weight;
  float ss = 0.f;
  if (F.gram) {
    ss = gram_row(F, th, c, iv * weight, gr, lane);
    if (gr) {   // the coordinates outside beta: zero, or the analytic sigma gradient
      for (int d = lane; d < Dtot; d += 32)
        if (d < beta_off || d >= beta_off + D) gr[d] = d == sigma_param ? weight * (ss * iv - (float)F.N) / sg : 0.f;
    }
    __syncwarp();
  } else {
    for (int t = lane; t < F.n_tiles; t += 32) ss += F.ss_part[(int64_t)t * Cp + c];
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  }
  float lp = F.logit ? weight * ss : weight * ((float)F.N * (-kHalfLog2Pi - logf(sg)) - 0.5f * ss * iv);
  // One warp per chain: with a scalar loop over d the warp walks D / 32 dependent iterations (80-120 us at D = 1000
  // whatever the number of chains: latency bound).  When the layout allows, each lane takes four consecutive
  // coefficients and all split-K partials of an iteration are independent 16-byte loads.
  const bool vec4 = !F.gram && gr && sigma_param < 0 && (Dtot & 3) == 0 && (beta_off & 3) == 0 && (D & 3) == 0 &&
                    ((reinterpret_cast<uintptr_t>(gr) | reinterpret_cast<uintptr_t>(G)) & 15) == 0;
  if (vec4) {
    const float ru = F.r_unscale ? F.r_unscale[c] : 1.0f;
    for (int d = 4 * lane; d < Dtot; d += 128) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (d >= beta_off && d < beta_off + D) {
        const float4 *g4 = reinterpret_cast<const float4 *>(G + (int64_t)c * Dp + (d - beta_off));
        const int64_t stride4 = (Cp * (int64_t)Dp) >> 2;
#pragma unroll 8
        for (int s = 0; s < F.g_splits; ++s) {   // fixed order, element by element the same sums as the scalar loop
          const float4 t = g4[(int64_t)s * stride4];
          v.x += t.x; v.y += t.y; v.z += t.z; v.w += t.w;
        }
        if (F.r_unscale) {
          const float4 ic = *reinterpret_cast<const float4 *>(F.inv_col_scale + (d - beta_off));
          v.x *= ru * ic.x; v.y *= ru * ic.y; v.z *= ru * ic.z; v.w *= ru * ic.w;
        }
      }
      *reinterpret_cast<float4 *>(gr + d) = v;
    }
    __syncwarp();
  } else if (gr && !F.gram) {
#pragma unroll 2
    for (int d = lane; d < Dtot; d += 32) {
      float v = 0.f;
      if (d >= beta_off && d < beta_off + D) {
#pragma unroll 8
        for (int s = 0; s < F.g_splits; ++s) v += G[((int64_t)s * Cp + c) * Dp + (d - beta_off)];  // fixed order
        if (F.r_unscale) v *= F.r_unscale[c] * F.inv_col_scale[d - beta_off];   // fp16 encoding: undo the operand scales
      }
      if (d == sigma_param) v = weight * (ss * iv - (float)F.N) / sg;
      gr[d] = v;
    }
    __syncwarp();
  }
  // priors: lanes stride the elements of each term; each element touches its own theta entries
  float pl = 0.f;
  const int n_terms = F.has_prior ? sm.n_terms : 0;
  for (int t = 0; t < n_terms; ++t) {
    const b2m_term &T = sm.terms[t];
    float acc = 0.f, ax = 0.f, a0 = 0.f, a1 = 0.f;
    if (T.dist == B2M_NORMAL && T.x.kind == B2M_OP_PARAMVEC && T.p0.kind == B2M_OP_CONST && T.p1.kind == B2M_OP_CONST) {
      // the usual coefficient prior, sum Normal(loc, scale).log_prob(beta): constants hoisted out of the element loop
      // (same expressions as dist_eval, evaluated once)
      const float p0 = T.p0.c, p1 = T.p1.c, var = p1 * p1, base = -kHalfLog2Pi - logf(p1), w = T.weight;
      const float *__restrict__ xv = th + T.x.a;
      float *__restrict__ gv = gr ? gr + T.x.a : nullptr;
      if ((T.length & 3) == 0 && ((reinterpret_cast<uintptr_t>(xv) | reinterpret_cast<uintptr_t>(gv)) & 15) == 0) {
        for (int n = 4 * lane; n < T.length; n += 128) {   // same per-element expressions, four elements per lane
          const float4 x4 = *reinterpret_cast<const float4 *>(xv + n);
          const float z0 = x4.x - p0, z1 = x4.y - p0, z2 = x4.z - p0, z3 = x4.w - p0;
          acc += base - (0.5f * (z0 * z0)) / var;
          acc += base - (0.5f * (z1 * z1)) / var;
          acc += base - (0.5f * (z2 * z2)) / var;
          acc += base - (0.5f * (z3 * z3)) / var;
          if (gv) {
            float4 g4 = *reinterpret_cast<float4 *>(gv + n);
            g4.x += w * (-(z0 / var)); g4.y += w * (-(z1 / var)); g4.z += w * (-(z2 / var)); g4.w += w * (-(z3 / var));
            *reinterpret_cast<float4 *>(gv + n) = g4;
          }
        }
      } else {
#pragma unroll 4
        for (int n = lane; n < T.length; n += 32) {
          const float z = xv[n] - p0;
          acc += base - (0.5f * (z * z)) / var;
          if (gv) gv[n] += w * (-(z / var));
        }
      }
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      pl += w * acc;
      __syncwarp();
      continue;
    }
    for (int n = lane; n < T.length; n += 32) {
      const float x = op_fetch(T.x, n, th, 1, sm), p0 = op_fetch(T.p0, n, th, 1, sm), p1 = op_fetch(T.p1, n, th, 1, sm);
      Elem e = dist_eval<true>(T.dist, x, p0, p1, T.k0, T.k1, T.k2);
      acc += e.lp;
      if (gr) {
        if (T.x.kind == B2M_OP_PARAM) ax += e.dx; else if (T.x.kind == B2M_OP_PARAMVEC) gr[T.x.a + n] += T.weight * e.dx;
        if (T.p0.kind == B2M_OP_PARAM) a0 += e.d0; else if (T.p0.kind == B2M_OP_PARAMVEC) gr[T.p0.a + n] += T.weight * e.d0;
        if (T.p1.kind == B2M_OP_PARAM) a1 += e.d1; else if (T.p1.kind == B2M_OP_PARAMVEC) gr[T.p1.a + n] += T.weight * e.d1;
      }
    }
    for (int o = 16; o > 0; o >>= 1) {
      acc += __shfl_xor_sync(0xffffffffu, acc, o);
      ax += __shfl_xor_sync(0xffffffffu, ax, o);
      a0 += __shfl_xor_sync(0xffffffffu, a0, o);
      a1 += __shfl_xor_sync(0xffffffffu, a1, o);
    }
    pl += T.weight * acc;
    if (gr && lane == 0) {
      if (T.x.kind == B2M_OP_PARAM) gr[T.x.a] += T.weight * ax;
      if (T.p0.kind == B2M_OP_PARAM) gr[T.p0.a] += T.weight * a0;
      if (T.p1.kind == B2M_OP_PARAM) gr[T.p1.a] += T.weight * a1;
    }
    __syncwarp();
  }
  float lj = 0.f;
  if (F.tf) {   // chain rule through theta = T(u) and the log-Jacobian
    for (int d = lane; d < Dtot; d += 32) {
      const int k = F.tf[d];
      if (k == B2M_TF_NONE) continue;
      const Tf t = tf_apply(k, thu[d]);
      lj += t.logjac;
      if (gr) gr[d] = fmaf(gr[d], t.jac, t.dlogjac);
    }
    for (int o = 16; o > 0; o >>= 1) lj += __shfl_xor_sync(0xffffffffu, lj, o);
    __syncwarp();
  }
  if (lane == 0) *logp_out = lp + pl + lj;
}

// host-side parameter blocks for the current state of a model (glm.cu)
PackP make_pack(const GlmModel &g);
FinishP make_finish(const GlmModel &g, int64_t Cp, bool with_grad);
size_t finish_smem(const GlmModel &g);

}  // namespace b2m

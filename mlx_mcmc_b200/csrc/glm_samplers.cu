// Lock-step samplers for GLM-class models: chain state lives in HBM as [C, Dtot] arrays, every leapfrog
// step of every chain shares one pair of dense contractions (glm_logp_grad), and small per-chain kernels
// (one warp per chain) do the integrator arithmetic, energies, U-turn dot products and tree bookkeeping.
//
// Replaces the same reference code as the pointwise kernels: kernels/hmc.py:113-198, kernels/nuts.py:137-343,
// kernels/metropolis.py:64-92.  The NUTS tree is the iterative restatement of build_tree (SURVEY.md 7a): one
// leaf per lock-step, per-chain masks for chains whose subtree / trajectory has ended.
#include <stdlib.h>

#include <chrono>
#include <string>
#include <vector>

#include "glm_rows.cuh"

namespace b2m {

constexpr int WPB = 4;  // warps (= chains) per block

__device__ __forceinline__ float warp_sum(float v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// N(0,1) for dimension d of (chain, iteration) -- same slot map as the pointwise kernels (common.cuh)
__device__ __forceinline__ void normals4(uint64_t seed, uint64_t gchain, uint32_t giter, int group, float out[4]) {
  // group 0 -> dims 2..5, group k -> dims 2+4k .. 5+4k (slot 1+k)
  const uint4 w = Philox::draw(seed, gchain, giter, 1u + (uint32_t)group);
  box_muller(w.x, w.y, out[0], out[1]);
  box_muller(w.z, w.w, out[2], out[3]);
}

// im = diag(M^-1) shared by all chains or nullptr (identity, the reference): p = z sqrt(m_d) ~ N(0, M)
// (__noinline__ on the vector helpers: the fused state kernel inlined ~35 copies of them into 24,000 instructions =
// 390 KB of code, and with a handful of warps per SM the kernel was bound by instruction-cache misses -- ncu: "no
// instruction" was the largest stall reason at the 1024-chain configuration.  They take plain pointers and scalars, so a
// call costs a few dozen cycles against the ~500-cycle memory round trips they contain.)
__device__ __noinline__ void fill_momentum(float *p, int D, const float *inj, uint64_t seed, uint64_t gchain, uint32_t giter,
                                           uint4 w0, int lane, const float *__restrict__ im = nullptr) {
  if (inj) {
    for (int d = lane; d < D; d += 32) p[d] = im ? inj[d] / sqrtf(im[d]) : inj[d];
    return;
  }
  if (lane == 0) {
    float a, b;
    box_muller(w0.x, w0.y, a, b);
    p[0] = a;
    if (D > 1) p[1] = b;
  }
  for (int grp = lane; 2 + 4 * grp < D; grp += 32) {
    float z[4];
    normals4(seed, gchain, giter, grp, z);
    for (int i = 0; i < 4; ++i)
      if (2 + 4 * grp + i < D) p[2 + 4 * grp + i] = z[i];
  }
  if (im) {
    __syncwarp();
    for (int d = lane; d < D; d += 32) p[d] = p[d] / sqrtf(im[d]);
  }
}

__device__ __noinline__ float kinetic_w(const float *__restrict__ p, int D, int lane, const float *__restrict__ im = nullptr) {
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  int d = lane;
  if (im) {   // 0.5 sum p_d^2 / m_d
    for (; d < D; d += 32) s0 = fmaf(p[d] * p[d], im[d], s0);
    return 0.5f * warp_sum(s0);
  }
  for (; d + 96 < D; d += 128) {
    const float a = p[d], b = p[d + 32], c = p[d + 64], e = p[d + 96];
    s0 = fmaf(a, a, s0); s1 = fmaf(b, b, s1); s2 = fmaf(c, c, s2); s3 = fmaf(e, e, s3);
  }
  for (; d < D; d += 32) s0 = fmaf(p[d], p[d], s0);
  return 0.5f * warp_sum((s0 + s1) + (s2 + s3));
}

#define CHAIN_PROLOGUE(C)                                                        \
  const int lane = threadIdx.x & 31;                                             \
  const int64_t c = (int64_t)blockIdx.x * WPB + (threadIdx.x >> 5);              \
  if (c >= (C)) return;

// ================================================================= HMC
struct HmcBufs {
  float *p, *g, *qn, *gn, *lp, *lpn, *h0;
  const int *tf;   // constraint transforms of the model (draws are written constrained) or nullptr
};

// one warp writes a draw: the constrained value unless the call asks for the sampler's own coordinates
__device__ __forceinline__ void write_draw(float *__restrict__ dst, const float *__restrict__ q, int D, int lane,
                                           const int *__restrict__ tf) {
  for (int d = lane; d < D; d += 32) dst[d] = tf_constrain(tf[d], q[d]);
}

__global__ void __launch_bounds__(32 * WPB) hmc_begin_kernel(b2m_hmc_args A, HmcBufs W, int D, int it) {
  CHAIN_PROLOGUE(A.n_chains)
  const uint64_t gchain = (uint64_t)(A.chain_offset + c);
  const uint32_t giter = (uint32_t)(A.iter_offset + it);
  const size_t row = (size_t)it * A.n_chains + c;
  float *p = W.p + c * D, *qn = W.qn + c * D;
  const float *q = A.theta + c * D, *g = W.g + c * D;
  const uint4 w0 = Philox::draw(A.seed, gchain, giter, 0u);
  const float *__restrict__ im = A.inv_mass;
  fill_momentum(p, D, A.inj_normal ? A.inj_normal + row * D : nullptr, A.seed, gchain, giter, w0, lane, im);
  __syncwarp();
  const float kin = kinetic_w(p, D, lane, im);
  if (lane == 0) W.h0[c] = -W.lp[c] + kin;
  const double eps = A.step_size[c];
  const float he = (float)(0.5 * eps), fe = (float)eps;
  for (int d = lane; d < D; d += 32) {
    const float pv = __fadd_rn(p[d], __fmul_rn(he, g[d]));
    p[d] = pv;
    qn[d] = __fadd_rn(q[d], __fmul_rn(fe, im ? im[d] * pv : pv));
  }
}

// between two leapfrog steps: second half kick of step l, first half kick + drift of step l+1
__global__ void __launch_bounds__(32 * WPB) hmc_mid_kernel(b2m_hmc_args A, HmcBufs W, int D) {
  CHAIN_PROLOGUE(A.n_chains)
  float *p = W.p + c * D, *qn = W.qn + c * D;
  const float *gn = W.gn + c * D;
  const double eps = A.step_size[c];
  const float he = (float)(0.5 * eps), fe = (float)eps;
  const float *__restrict__ im = A.inv_mass;
  for (int d = lane; d < D; d += 32) {
    float pv = __fadd_rn(p[d], __fmul_rn(he, gn[d]));
    pv = __fadd_rn(pv, __fmul_rn(he, gn[d]));
    p[d] = pv;
    qn[d] = __fadd_rn(qn[d], __fmul_rn(fe, im ? im[d] * pv : pv));
  }
}

__global__ void __launch_bounds__(32 * WPB) hmc_end_kernel(b2m_hmc_args A, HmcBufs W, int D, int it) {
  CHAIN_PROLOGUE(A.n_chains)
  const uint64_t gchain = (uint64_t)(A.chain_offset + c);
  const uint32_t giter = (uint32_t)(A.iter_offset + it);
  const size_t row = (size_t)it * A.n_chains + c;
  float *p = W.p + c * D, *q = A.theta + c * D, *g = W.g + c * D;
  const float *qn = W.qn + c * D, *gn = W.gn + c * D;
  double eps = A.step_size[c];
  const float he = (float)(0.5 * eps);
  for (int d = lane; d < D; d += 32) p[d] = __fadd_rn(p[d], __fmul_rn(he, gn[d]));
  __syncwarp();
  const float kin = kinetic_w(p, D, lane, A.inv_mass);
  const float h0 = W.h0[c], h1 = -W.lpn[c] + kin;
  float u;
  if (A.inj_uniform) u = A.inj_uniform[row];
  else u = u01(Philox::draw(A.seed, gchain, giter, 0u).z);
  const float log_ratio = -(h1 - h0);
  const bool accept = logf(u) < log_ratio;
  if (accept) {
    for (int d = lane; d < D; d += 32) { q[d] = qn[d]; g[d] = gn[d]; }
  }
  if (lane == 0) {
    if (accept) W.lp[c] = W.lpn[c];
    int64_t n_acc = A.n_accept[c] + (accept ? 1 : 0), n_tot = A.n_total[c] + 1;
    A.n_accept[c] = n_acc;
    A.n_total[c] = n_tot;
    if (A.adapt == B2M_ADAPT_REFERENCE) {
      if ((int64_t)giter > 10) eps *= ((double)n_acc / (double)n_tot < A.target_accept) ? 0.95 : 1.05;
      A.step_size[c] = eps;
    } else if (A.adapt == B2M_ADAPT_DUAL_AVERAGING) {
      double h_bar = A.da_state[c * 3 + 0], log_eps_bar = A.da_state[c * 3 + 1];
      const double mu = A.da_state[c * 3 + 2];
      const float a = (log_ratio == log_ratio) ? expf(fminf(log_ratio, 0.f)) : 0.f;
      const double m = (double)((int64_t)giter - A.adapt_origin) + 1.0, eta = 1.0 / (m + 10.0);
      h_bar = (1.0 - eta) * h_bar + eta * (A.target_accept - (double)a);
      double log_eps = mu - sqrt(m) / 0.05 * h_bar;
      log_eps = fmin(fmax(log_eps, -10.0), 10.0);
      const double wt = pow(m, -0.75);
      log_eps_bar = wt * log_eps + (1.0 - wt) * log_eps_bar;
      A.step_size[c] = exp(log_eps);
      A.da_state[c * 3 + 0] = h_bar;
      A.da_state[c * 3 + 1] = log_eps_bar;
    }
    if (A.trace_energy) { A.trace_energy[row * 2] = h0; A.trace_energy[row * 2 + 1] = h1; }
    if (A.trace_accept) A.trace_accept[row] = accept ? 1 : 0;
  }
  if (A.draws) {
    __syncwarp();
    if (W.tf && !A.draws_unconstrained) write_draw(A.draws + row * D, q, D, lane, W.tf);
    else for (int d = lane; d < D; d += 32) A.draws[row * D + d] = q[d];
  }
}

// Workspace: carved from one arena owned by the model handle and reused across calls (a sampler call per
// iteration must not pay for dozens of cudaMalloc / cudaFree).  `take` is run twice: once on an empty arena to
// measure, once on the real one to assign.
struct Arena {
  char *base = nullptr;
  size_t off = 0;
  template <typename T>
  void take(T **p, size_t n) {
    off = (off + 255) & ~size_t(255);
    *p = base ? reinterpret_cast<T *>(base + off) : nullptr;
    off += sizeof(T) * (n ? n : 1);
  }
};

static int arena_reserve(GlmModel &g, size_t bytes) {
  if (bytes > g.ws_cap) {
    if (g.ws) cudaFree(g.ws);
    g.ws = nullptr;
    g.ws_cap = 0;
    B2M_CHECK_CUDA(cudaMalloc(reinterpret_cast<void **>(&g.ws), bytes));
    g.ws_cap = bytes;
  }
  if (!g.h_flag) {
    B2M_CHECK_CUDA(cudaMallocHost(reinterpret_cast<void **>(&g.h_flag), sizeof(int) * 16));
    g.h_ring = g.h_flag + 4;   // 8-byte aligned ring of four 64-bit counters
  }
  return 0;
}

int glm_hmc_run(GlmModel &gm, const b2m_hmc_args &a, cudaStream_t st) {
  const int64_t C = a.n_chains;
  const int D = gm.Dtot;
  HmcBufs W{};
  W.tf = gm.tf;
  auto layout = [&](Arena &A) {
    A.take(&W.p, C * D); A.take(&W.g, C * D); A.take(&W.qn, C * D); A.take(&W.gn, C * D);
    A.take(&W.lp, C); A.take(&W.lpn, C); A.take(&W.h0, C);
  };
  Arena probe;
  layout(probe);
  if (int rc0 = arena_reserve(gm, probe.off)) return rc0;
  Arena real;
  real.base = gm.ws;
  layout(real);
  const unsigned grid = (unsigned)((C + WPB - 1) / WPB);
  int rc = glm_logp_grad(gm, a.theta, C, W.lp, W.g, st, true);
  for (int it = 0; it < a.n_iter && !rc; ++it) {
    if (it > 0) rc = glm_recenter(gm, a.theta, C, st);   // reference point follows the current states
    hmc_begin_kernel<<<grid, 32 * WPB, 0, st>>>(a, W, D, it);
    ++g_launches;
    for (int l = 0; l < a.n_leapfrog && !rc; ++l) {
      rc = glm_logp_grad(gm, W.qn, C, W.lpn, W.gn, st);
      if (l + 1 < a.n_leapfrog) {
        hmc_mid_kernel<<<grid, 32 * WPB, 0, st>>>(a, W, D);
        ++g_launches;
      }
    }
    hmc_end_kernel<<<grid, 32 * WPB, 0, st>>>(a, W, D, it);
    ++g_launches;
  }
  cudaError_t e = cudaStreamSynchronize(st);
  if (rc) return rc;
  B2M_CHECK_CUDA(e);
  B2M_CHECK_CUDA(cudaGetLastError());
  return 0;
}

// ================================================================= Metropolis
__global__ void __launch_bounds__(32 * WPB) mh_propose_kernel(b2m_mh_args A, float *qn, int D, int it) {
  CHAIN_PROLOGUE(A.n_chains)
  const uint64_t gchain = (uint64_t)(A.chain_offset + c);
  const uint32_t giter = (uint32_t)(A.iter_offset + it);
  const size_t row = (size_t)it * A.n_chains + c;
  float *z = qn + c * D;
  const float *q = A.theta + c * D;
  const uint4 w0 = Philox::draw(A.seed, gchain, giter, 0u);
  fill_momentum(z, D, A.inj_normal ? A.inj_normal + row * D : nullptr, A.seed, gchain, giter, w0, lane);
  __syncwarp();
  for (int d = lane; d < D; d += 32) z[d] = __fadd_rn(q[d], __fmul_rn(z[d], A.proposal_scale));
}

__global__ void __launch_bounds__(32 * WPB) mh_accept_kernel(b2m_mh_args A, const float *qn, const float *lpn, int D, int it,
                                                             const int *__restrict__ tf) {
  CHAIN_PROLOGUE(A.n_chains)
  const uint64_t gchain = (uint64_t)(A.chain_offset + c);
  const uint32_t giter = (uint32_t)(A.iter_offset + it);
  const size_t row = (size_t)it * A.n_chains + c;
  float *q = A.theta + c * D;
  float u;
  if (A.inj_uniform) u = A.inj_uniform[row];
  else u = u01(Philox::draw(A.seed, gchain, giter, 0u).z);
  const bool accept = logf(u) < __fsub_rn(lpn[c], A.logp[c]);
  if (accept)
    for (int d = lane; d < D; d += 32) q[d] = qn[c * D + d];
  __syncwarp();
  if (lane == 0) {
    if (accept) { A.logp[c] = lpn[c]; A.n_accept[c] += 1; }
    if (A.trace_accept) A.trace_accept[row] = accept ? 1 : 0;
  }
  if (A.draws) {
    if (tf) write_draw(A.draws + row * D, q, D, lane, tf);
    else for (int d = lane; d < D; d += 32) A.draws[row * D + d] = q[d];
  }
}

int glm_mh_run(GlmModel &gm, const b2m_mh_args &a, cudaStream_t st) {
  const int64_t C = a.n_chains;
  const int D = gm.Dtot;
  float *qn = nullptr, *lpn = nullptr;
  auto layout = [&](Arena &A) { A.take(&qn, C * D); A.take(&lpn, C); };
  Arena probe;
  layout(probe);
  if (int rc0 = arena_reserve(gm, probe.off)) return rc0;
  Arena real;
  real.base = gm.ws;
  layout(real);
  const unsigned grid = (unsigned)((C + WPB - 1) / WPB);
  // the cached current log-prob is recomputed at the start of every call, as metropolis.py:55 does
  int rc = glm_logp_grad(gm, a.theta, C, a.logp, nullptr, st, true);
  for (int it = 0; it < a.n_iter && !rc; ++it) {
    if (it > 0 && (it & 15) == 0) rc = glm_recenter(gm, a.theta, C, st);
    mh_propose_kernel<<<grid, 32 * WPB, 0, st>>>(a, qn, D, it);
    rc = glm_logp_grad(gm, qn, C, lpn, nullptr, st);
    mh_accept_kernel<<<grid, 32 * WPB, 0, st>>>(a, qn, lpn, D, it, gm.tf);
    g_launches += 2;
  }
  cudaError_t e = cudaStreamSynchronize(st);
  if (rc) return rc;
  B2M_CHECK_CUDA(e);
  B2M_CHECK_CUDA(cudaGetLastError());
  return 0;
}

// ================================================================= NUTS
struct NutsBufs {
  // [C, D] vectors: gradient at the starting points of the call, and the working leaf (position, momentum, gradient)
  float *g, *fq, *fp, *fg;
  // Saved tree states: n_slots slots per chain, [C, n_slots, 3, D]; slot s of chain c holds q, p, g as three [D] rows.
  // The tree refers to them by per-chain slot numbers, so a merge, a push or a candidate choice moves an index, not a
  // vector.  Live at once: lo, hi, cand and st_f / st_c of every parked level (at most 2 MD + 1), plus the new leaf.
  float *slots;
  int n_slots;
  int *lo, *hi, *cand;   // [C] trajectory edges and the candidate
  int *leaf_slot;        // [C] the last completed leaf (the start of the next leaf; the new edge at a doubling's end)
  int *sub_c;            // [C] candidate of the completed subtree of the current doubling
  int *st_f, *st_c;      // [MD, C] first edge and candidate of the parked left subtrees
  // [C] scalars
  float *lp, *clp, *h0, *log_slice, *flp, *sclp, *feps, *heps;
  int *n, *s, *v, *leaf, *building, *sub_n, *sub_na, *sub_s, *alpha_cnt, *depth;
  double *alpha_sum, *sub_alpha;
  // [MD, C] stack scalars
  float *st_clp;
  int *st_n, *st_na;
  double *st_alpha;
  int *n_active;    // device: number of chains building in the current doubling
  int *active;      // [C] ordered list of those chains (the compacted lock-step batch)
  float *alpha_it;  // [C] this iteration's mean acceptance statistic (pooled adaptation)
  double *eps_it;   // [C] step size of this iteration (= step_size, or its jittered value)
  // iteration-asynchronous schedule (glm_nuts_run_async)
  int *state;       // [C] 0 = not started, 1 = a leaf is being evaluated, 2 = all iterations done
  int *iter;        // [C] the chain's own iteration counter
  int *fin;         // [C] finished an iteration in the current tick (pooled adaptation)
  int *live;        // [C] state != 2 (input of the compaction)
  int *n_done;      // device counter of finished chains
  double *pool;     // [4] pooled adaptation: sum of alpha, count, update index, spare
  const int *tf;    // constraint transforms of the model (draws are written constrained) or nullptr
};

// One warp copies a [D] vector.  These kernels are pure HBM streaming with one warp per chain: with a scalar loop each
// lane has a single 4-byte load in flight and the copy is latency bound (the v1 leaf kernels took 120-200 us for
// ~300 MB of traffic); 16-byte accesses, four independent loads before the first store, put enough bytes in flight.
__device__ __noinline__ void vcopy(float *__restrict__ dst, const float *__restrict__ src, int D, int lane) {
  if ((D & 3) == 0 && ((reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src)) & 15) == 0) {
    const float4 *__restrict__ s4 = reinterpret_cast<const float4 *>(src);
    float4 *__restrict__ d4 = reinterpret_cast<float4 *>(dst);
    const int n4 = D >> 2;
    for (int i = lane; i < n4; i += 128) {   // up to four predicated 16-byte loads in flight per lane
      const bool pb = i + 32 < n4, pc = i + 64 < n4, pe = i + 96 < n4;
      float4 a = s4[i], b = a, c = a, e = a;
      if (pb) b = s4[i + 32];
      if (pc) c = s4[i + 64];
      if (pe) e = s4[i + 96];
      d4[i] = a;
      if (pb) d4[i + 32] = b;
      if (pc) d4[i + 64] = c;
      if (pe) d4[i + 96] = e;
    }
  } else {
    for (int d = lane; d < D; d += 128) {
      const bool pb = d + 32 < D, pc = d + 64 < D, pe = d + 96 < D;
      float a = src[d], b = 0.f, c = 0.f, e = 0.f;
      if (pb) b = src[d + 32];
      if (pc) c = src[d + 64];
      if (pe) e = src[d + 96];
      dst[d] = a;
      if (pb) dst[d + 32] = b;
      if (pc) dst[d + 64] = c;
      if (pe) dst[d + 96] = e;
    }
  }
}

// continue-straight test of nuts.py:119-135 on [D] vectors (warp reduction)
__device__ __noinline__ bool straight_w(const float *q_lo, const float *q_hi, const float *p_lo, const float *p_hi,
                                        int D, int lane) {
  float a = 0.f, b = 0.f;
#pragma unroll 4
  for (int d = lane; d < D; d += 32) {
    const float dq = q_hi[d] - q_lo[d];
    a = fmaf(dq, p_lo[d], a);
    b = fmaf(dq, p_hi[d], b);
  }
  a = warp_sum(a);
  b = warp_sum(b);
  return a >= 0.f && b >= 0.f;
}

// row r (0 = q, 1 = p, 2 = g) of slot s of chain c
__device__ __forceinline__ float *slot_row(const NutsBufs &W, int D, int64_t c, int s, int r) {
  return W.slots + (((size_t)c * W.n_slots + s) * 3 + r) * D;
}

__device__ __forceinline__ void nuts_begin_dev(const b2m_nuts_args &A, const NutsBufs &W, int D, int64_t c, int lane, int it) {
  const uint64_t gchain = (uint64_t)(A.chain_offset + c);
  const uint32_t giter = (uint32_t)(A.iter_offset + it);
  const size_t row = (size_t)it * A.n_chains + c;
  const size_t o = (size_t)c * D;
  const uint4 w0 = Philox::draw(A.seed, gchain, giter, 0u);
  // the start slot: the previous transition's candidate already holds theta and its gradient; the first transition
  // of a call takes them from the caller's theta and the gradient evaluated at the start of the call
  int s0 = 0;
  if (it == 0) {
    vcopy(slot_row(W, D, c, 0, 0), A.theta + o, D, lane);
    vcopy(slot_row(W, D, c, 0, 2), W.g + o, D, lane);
  } else {
    s0 = W.cand[c];
  }
  float *p = slot_row(W, D, c, s0, 1);
  fill_momentum(p, D, A.inj_normal ? A.inj_normal + row * D : nullptr, A.seed, gchain, giter, w0, lane, A.inv_mass);
  __syncwarp();
  const float kin = kinetic_w(p, D, lane, A.inv_mass);
  if (lane == 0) {
    W.lo[c] = s0; W.hi[c] = s0; W.cand[c] = s0;
    const float h0 = -W.lp[c] + kin;
    const float us = A.inj_slice ? A.inj_slice[row] : u01(w0.z);
    const double log_u64 = (double)(-h0) + (double)logf(us);
    W.h0[c] = h0;
    W.log_slice[c] = A.compat == B2M_COMPAT_REFERENCE ? logf(expf((float)log_u64)) : (float)log_u64;
    W.clp[c] = W.lp[c];
    W.n[c] = 1; W.s[c] = 1; W.alpha_sum[c] = 0.0; W.alpha_cnt[c] = 0; W.depth[c] = 0; W.building[c] = 0;
    const double eps = A.step_size[c];
    W.eps_it[c] = A.step_size_jitter > 0.f ? eps * (1.0 + (double)A.step_size_jitter * (2.0 * (double)u01(w0.w) - 1.0)) : eps;
    if (A.trace_energy) A.trace_energy[row] = h0;
  }
}

__global__ void __launch_bounds__(32 * WPB) nuts_begin_kernel(b2m_nuts_args A, NutsBufs W, int D, int it) {
  CHAIN_PROLOGUE(A.n_chains)
  nuts_begin_dev(A, W, D, c, lane, it);
}

__device__ __forceinline__ void nuts_doubling_begin_dev(const b2m_nuts_args &A, const NutsBufs &W, int D, int64_t c, int lane, int it, int j) {
  if (!W.s[c]) { if (lane == 0) W.building[c] = 0; return; }
  const uint64_t gchain = (uint64_t)(A.chain_offset + c);
  const uint32_t giter = (uint32_t)(A.iter_offset + it);
  const size_t row = (size_t)it * A.n_chains + c;
  float ud;
  if (A.inj_dir) ud = A.inj_dir[row * A.max_tree_depth + j];
  else ud = u01(Philox::draw(A.seed, gchain, giter, SLOT_NUTS_DOUBLING + j).x);
  const int v = ud < 0.5f ? 1 : -1;
  if (lane == 0) {
    const double eps = W.eps_it[c];
    W.leaf_slot[c] = v == 1 ? W.hi[c] : W.lo[c];   // the first leaf steps off the edge in direction v
    W.v[c] = v;
    W.feps[c] = (float)((double)v * eps);
    W.heps[c] = (float)(0.5 * ((double)v * eps));
    W.leaf[c] = 0;
    W.building[c] = 1;
  }
}

__global__ void __launch_bounds__(32 * WPB) nuts_doubling_begin_kernel(b2m_nuts_args A, NutsBufs W, int D, int it, int j) {
  CHAIN_PROLOGUE(A.n_chains)
  nuts_doubling_begin_dev(A, W, D, c, lane, it, j);
}

__device__ __forceinline__ void nuts_leaf_pre_dev(const b2m_nuts_args &A, const NutsBufs &W, int D, int64_t c, int lane) {
  if (!W.building[c]) return;
  const size_t o = (size_t)c * D;
  const float he = W.heps[c], fe = W.feps[c];
  float *__restrict__ fq = W.fq + o, *__restrict__ fp = W.fp + o;
  // start state: the last leaf, or the edge the doubling extends
  const int s = W.leaf_slot[c];
  const float *__restrict__ sq = slot_row(W, D, c, s, 0), *__restrict__ sp = slot_row(W, D, c, s, 1),
                            *__restrict__ sg = slot_row(W, D, c, s, 2);
  if (const float *__restrict__ im = A.inv_mass) {   // diagonal mass matrix: drift by eps M^-1 p
#pragma unroll 4
    for (int d = lane; d < D; d += 32) {
      const float pv = __fadd_rn(sp[d], __fmul_rn(he, sg[d]));
      fp[d] = pv;
      fq[d] = __fadd_rn(sq[d], __fmul_rn(fe, im[d] * pv));
    }
    return;
  }
  if ((D & 3) == 0 && ((reinterpret_cast<uintptr_t>(fq) | reinterpret_cast<uintptr_t>(fp) | reinterpret_cast<uintptr_t>(sq) |
                        reinterpret_cast<uintptr_t>(sp) | reinterpret_cast<uintptr_t>(sg)) & 15) == 0) {
    for (int d = 4 * lane; d < D; d += 128) {   // four coefficients per lane: same per-element arithmetic
      const float4 g4 = *reinterpret_cast<const float4 *>(sg + d);
      float4 p4 = *reinterpret_cast<const float4 *>(sp + d), q4 = *reinterpret_cast<const float4 *>(sq + d);
      p4.x = __fadd_rn(p4.x, __fmul_rn(he, g4.x)); p4.y = __fadd_rn(p4.y, __fmul_rn(he, g4.y));
      p4.z = __fadd_rn(p4.z, __fmul_rn(he, g4.z)); p4.w = __fadd_rn(p4.w, __fmul_rn(he, g4.w));
      q4.x = __fadd_rn(q4.x, __fmul_rn(fe, p4.x)); q4.y = __fadd_rn(q4.y, __fmul_rn(fe, p4.y));
      q4.z = __fadd_rn(q4.z, __fmul_rn(fe, p4.z)); q4.w = __fadd_rn(q4.w, __fmul_rn(fe, p4.w));
      *reinterpret_cast<float4 *>(fp + d) = p4;
      *reinterpret_cast<float4 *>(fq + d) = q4;
    }
    return;
  }
#pragma unroll 4
  for (int d = lane; d < D; d += 32) {
    const float pv = __fadd_rn(sp[d], __fmul_rn(he, sg[d]));
    fp[d] = pv;
    fq[d] = __fadd_rn(sq[d], __fmul_rn(fe, pv));
  }
}

__global__ void __launch_bounds__(32 * WPB) nuts_leaf_pre_kernel(b2m_nuts_args A, NutsBufs W, int D) {
  CHAIN_PROLOGUE(A.n_chains)
  nuts_leaf_pre_dev(A, W, D, c, lane);
}

__device__ __forceinline__ void nuts_leaf_post_dev(const b2m_nuts_args &A, const NutsBufs &W, int D, int64_t c, int lane, int it, int j) {
  if (!W.building[c]) return;
  const int64_t C = A.n_chains;
  const uint64_t gchain = (uint64_t)(A.chain_offset + c);
  const uint32_t giter = (uint32_t)(A.iter_offset + it);
  const size_t row = (size_t)it * C + c;
  const size_t o = (size_t)c * D;
  const int MD = A.max_tree_depth;
  const bool ref_compat = A.compat == B2M_COMPAT_REFERENCE;
  const float *fq = W.fq + o, *fp = W.fp + o, *fg = W.fg + o;
  const float he = W.heps[c];
  const int i = W.leaf[c];
  // a free slot for this leaf: one that is not an edge, not the candidate and not a parked subtree (the parked levels
  // are the set bits of the leaf index)
  unsigned live = (1u << W.lo[c]) | (1u << W.hi[c]) | (1u << W.cand[c]);
  for (int k = 0; k < j; ++k)
    if ((i >> k) & 1) live |= (1u << W.st_f[(size_t)k * C + c]) | (1u << W.st_c[(size_t)k * C + c]);
  const int L = __ffs(~live) - 1;
  B2M_ASSERT(L >= 0 && L < W.n_slots);
  float *__restrict__ lq = slot_row(W, D, c, L, 0), *__restrict__ lp = slot_row(W, D, c, L, 1), *__restrict__ lg = slot_row(W, D, c, L, 2);
  // one pass: second half kick, kinetic energy, and the completed leaf stored into its slot -- three loads and three
  // stores per element.  The leaf is then both the first edge and the candidate of the subtree being assembled.
  float k0 = 0.f, k1 = 0.f;
  {
    int d = lane;
    if ((D & 3) == 0 && ((reinterpret_cast<uintptr_t>(fq) | reinterpret_cast<uintptr_t>(fp) | reinterpret_cast<uintptr_t>(fg) |
                          reinterpret_cast<uintptr_t>(lq) | reinterpret_cast<uintptr_t>(lp) | reinterpret_cast<uintptr_t>(lg)) & 15) == 0) {
      for (int e = 4 * lane; e < D; e += 128) {   // four coefficients per lane
        const float4 q4 = *reinterpret_cast<const float4 *>(fq + e), g4 = *reinterpret_cast<const float4 *>(fg + e);
        float4 p4 = *reinterpret_cast<const float4 *>(fp + e);
        p4.x = __fadd_rn(p4.x, __fmul_rn(he, g4.x)); p4.y = __fadd_rn(p4.y, __fmul_rn(he, g4.y));
        p4.z = __fadd_rn(p4.z, __fmul_rn(he, g4.z)); p4.w = __fadd_rn(p4.w, __fmul_rn(he, g4.w));
        k0 = fmaf(p4.x, p4.x, k0); k1 = fmaf(p4.y, p4.y, k1); k0 = fmaf(p4.z, p4.z, k0); k1 = fmaf(p4.w, p4.w, k1);
        *reinterpret_cast<float4 *>(lq + e) = q4; *reinterpret_cast<float4 *>(lp + e) = p4; *reinterpret_cast<float4 *>(lg + e) = g4;
      }
      d = D;   // nothing left for the scalar loops
    }
    for (; d + 32 < D; d += 64) {
      const float q0 = fq[d], q1 = fq[d + 32], g0 = fg[d], g1 = fg[d + 32];
      const float p0 = __fadd_rn(fp[d], __fmul_rn(he, g0)), p1 = __fadd_rn(fp[d + 32], __fmul_rn(he, g1));
      k0 = fmaf(p0, p0, k0); k1 = fmaf(p1, p1, k1);
      lq[d] = q0; lq[d + 32] = q1; lp[d] = p0; lp[d + 32] = p1; lg[d] = g0; lg[d + 32] = g1;
    }
    for (; d < D; d += 32) {
      const float q0 = fq[d], g0 = fg[d];
      const float p0 = __fadd_rn(fp[d], __fmul_rn(he, g0));
      k0 = fmaf(p0, p0, k0);
      lq[d] = q0; lp[d] = p0; lg[d] = g0;
    }
  }
  float kin = 0.5f * warp_sum(k0 + k1);
  __syncwarp();
  if (A.inv_mass) kin = kinetic_w(lp, D, lane, A.inv_mass);   // 0.5 sum p^2 / m (lp holds the completed step's momentum)
  const float flp = W.flp[c], h0 = W.h0[c], log_slice = W.log_slice[c];
  const float h1 = -flp + kin;
  const int n1 = (log_slice <= -h1) ? 1 : 0;
  const bool s1 = log_slice < (1000.0f - h1);
  float a1 = expf(-h1 + h0);
  if (a1 != a1) a1 = ref_compat ? 1.0f : 0.0f;
  a1 = fminf(a1, 1.0f);
  const int v = W.v[c];
  B2M_ASSERT(j >= 0 && j < A.max_tree_depth && i >= 0 && i < (1 << j) && (v == 1 || v == -1));
  if (lane == 0) {
    A.n_leaves[c] += 1;
    if (!s1) A.n_diverge[c] += 1;
  }
  float sub_clp = flp;
  int sub_n = n1, sub_na = 1;
  bool sub_s = s1;
  double sub_alpha = (double)a1;
  int sf = L, sc = L;   // first edge and candidate of the subtree being assembled
  int k = 0;
  bool finished = false;
  while (true) {
    if (k == j) { finished = true; break; }
    const size_t ss = (size_t)k * C + c;
    if ((i >> k) & 1) {
      const int m = i - __popc(i) + k;
      float um;
      if (A.inj_merge) {
        um = A.inj_merge[(row * MD + j) * ((1 << MD) - 1) + m];
      } else {
        const uint4 wm = Philox::draw(A.seed, gchain, giter, SLOT_NUTS_MERGE + 1024u * j + (m >> 2));
        const uint32_t word = (m & 3) == 0 ? wm.x : (m & 3) == 1 ? wm.y : (m & 3) == 2 ? wm.z : wm.w;
        um = u01(word);
      }
      const int n_tot = W.st_n[ss] + sub_n;
      const double ratio = (double)sub_n / fmax((double)n_tot, 1.0);
      if (!((double)um < ratio)) {
        sc = W.st_c[ss];
        sub_clp = W.st_clp[ss];
      }
      // the parked subtree's first edge against the far edge of this one (the leaf just stored)
      const int pf = W.st_f[ss];
      const float *fq_k = slot_row(W, D, c, pf, 0), *fp_k = slot_row(W, D, c, pf, 1);
      bool st;
      if (v == 1) st = straight_w(fq_k, lq, fp_k, lp, D, lane);
      else        st = straight_w(lq, fq_k, lp, fp_k, D, lane);
      sub_s = sub_s && st;
      sf = pf;
      sub_n = n_tot;
      sub_alpha = W.st_alpha[ss] + sub_alpha;
      sub_na = W.st_na[ss] + sub_na;
      ++k;
    } else {
      if (sub_s) {
        if (lane == 0) {
          W.st_f[ss] = sf; W.st_c[ss] = sc;
          W.st_clp[ss] = sub_clp; W.st_n[ss] = sub_n; W.st_na[ss] = sub_na; W.st_alpha[ss] = sub_alpha;
        }
        break;
      }
      ++k;
    }
  }
  if (lane == 0) {
    W.leaf_slot[c] = L;
    if (finished) {
      W.building[c] = 0;
      W.sub_c[c] = sc;
      W.sclp[c] = sub_clp; W.sub_n[c] = sub_n; W.sub_na[c] = sub_na; W.sub_s[c] = sub_s ? 1 : 0; W.sub_alpha[c] = sub_alpha;
    } else {
      W.leaf[c] = i + 1;
    }
  }
}

__global__ void __launch_bounds__(32 * WPB) nuts_leaf_post_kernel(b2m_nuts_args A, NutsBufs W, int D, int it, int j) {
  CHAIN_PROLOGUE(A.n_chains)
  nuts_leaf_post_dev(A, W, D, c, lane, it, j);
}

__device__ __forceinline__ void nuts_doubling_end_dev(const b2m_nuts_args &A, const NutsBufs &W, int D, int64_t c, int lane, int it, int j) {
  if (!W.s[c]) return;  // chain was not growing in this doubling
  const uint64_t gchain = (uint64_t)(A.chain_offset + c);
  const uint32_t giter = (uint32_t)(A.iter_offset + it);
  const size_t row = (size_t)it * A.n_chains + c;
  const int v = W.v[c];
  int lo = W.lo[c], hi = W.hi[c];
  if (v == 1) hi = W.leaf_slot[c];   // the last leaf is the new edge in direction v
  else        lo = W.leaf_slot[c];
  const int sub_n = W.sub_n[c], sub_s = W.sub_s[c];
  const int n = W.n[c];
  int took = 0;
  if (sub_s) {
    float ut;
    if (A.inj_take) ut = A.inj_take[row * A.max_tree_depth + j];
    else ut = u01(Philox::draw(A.seed, gchain, giter, SLOT_NUTS_DOUBLING + j).y);
    const double pr = fmin(1.0, (double)sub_n / fmax((double)n, 1.0));
    if ((double)ut < pr) took = 1;
  }
  const bool st = straight_w(slot_row(W, D, c, lo, 0), slot_row(W, D, c, hi, 0), slot_row(W, D, c, lo, 1),
                             slot_row(W, D, c, hi, 1), D, lane);
  const int s_new = (sub_s && st) ? 1 : 0;
  if (lane == 0) {
    W.lo[c] = lo; W.hi[c] = hi;
    if (took) { W.cand[c] = W.sub_c[c]; W.clp[c] = W.sclp[c]; }
    W.n[c] = n + sub_n;
    W.s[c] = s_new;
    W.alpha_sum[c] += W.sub_alpha[c];
    W.alpha_cnt[c] += W.sub_na[c];
    W.depth[c] = j + 1;
    if (A.trace_doubling) {
      int32_t *tr = A.trace_doubling + ((size_t)row * A.max_tree_depth + j) * 6;
      tr[0] = v; tr[1] = sub_n; tr[2] = sub_s; tr[3] = took; tr[4] = s_new; tr[5] = n + sub_n;
    }
  }
}

__global__ void __launch_bounds__(32 * WPB) nuts_doubling_end_kernel(b2m_nuts_args A, NutsBufs W, int D, int it, int j) {
  CHAIN_PROLOGUE(A.n_chains)
  nuts_doubling_end_dev(A, W, D, c, lane, it, j);
}

__device__ __forceinline__ void nuts_end_dev(const b2m_nuts_args &A, const NutsBufs &W, int D, int64_t c, int lane, int it) {
  const uint32_t giter = (uint32_t)(A.iter_offset + it);
  const size_t row = (size_t)it * A.n_chains + c;
  // the candidate slot stays as it is: the next transition starts from it (nuts_begin_dev)
  const float *cq = slot_row(W, D, c, W.cand[c], 0);
  vcopy(A.theta + (size_t)c * D, cq, D, lane);
  if (A.draws) {
    if (W.tf && !A.draws_unconstrained) write_draw(A.draws + row * D, cq, D, lane, W.tf);
    else vcopy(A.draws + row * D, cq, D, lane);
  }
  if (lane == 0) {
    W.lp[c] = W.clp[c];
    const double mean_alpha = W.alpha_sum[c] / fmax((double)W.alpha_cnt[c], 1.0);
    A.n_accept[c] += mean_alpha > 0.5 ? 1 : 0;
    if (A.adapt == B2M_ADAPT_POOLED) W.alpha_it[c] = (float)mean_alpha;
    if (A.adapt == B2M_ADAPT_DUAL_AVERAGING) {
      double h_bar = A.da_state[c * 3 + 0], eps_bar = A.da_state[c * 3 + 1];
      const float mu = (float)A.da_state[c * 3 + 2];
      const double m = (double)((int64_t)giter - A.adapt_origin), eta = 1.0 / (m + 10.0);
      h_bar = (1.0 - eta) * h_bar + eta * (A.target_accept - mean_alpha);
      float log_eps = __fsub_rn(mu, (float)((sqrt(m + 1.0) / 0.05) * h_bar));
      log_eps = fmaxf(fminf(log_eps, 10.0f), -10.0f);
      const double eps = (double)expf(log_eps);
      const double wgt = pow(m + 1.0, -0.75);
      eps_bar = (double)expf((float)(wgt * log(eps) + (1.0 - wgt) * log(eps_bar)));
      A.step_size[c] = eps;
      A.da_state[c * 3 + 0] = h_bar;
      A.da_state[c * 3 + 1] = eps_bar;
    }
    if (A.depths) A.depths[row] = W.depth[c];
    if (A.alphas) A.alphas[row] = (float)mean_alpha;
  }
}

__global__ void __launch_bounds__(32 * WPB) nuts_end_kernel(b2m_nuts_args A, NutsBufs W, int D, int it) {
  CHAIN_PROLOGUE(A.n_chains)
  nuts_end_dev(A, W, D, c, lane, it);
}

// Ordered compaction of the chains still building in this doubling: active[0..n) = their ids, ascending.
// One block; the list drives the compacted lock-step evaluations (glm_logp_grad with idx).
__global__ void __launch_bounds__(1024) nuts_compact_kernel(const int *__restrict__ building, int64_t C,
                                                            int *__restrict__ active, int *__restrict__ n_active) {
  __shared__ int warp_tot[32];
  __shared__ int base;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) base = 0;
  __syncthreads();
  for (int64_t c0 = 0; c0 < C; c0 += 1024) {
    const int64_t c = c0 + threadIdx.x;
    const int f = (c < C && building[c]) ? 1 : 0;
    const unsigned bal = __ballot_sync(0xffffffffu, f);
    const int pre = __popc(bal & ((1u << lane) - 1u));
    if (lane == 0) warp_tot[warp] = __popc(bal);
    __syncthreads();
    int off = 0, tot = 0;
    for (int w = 0; w < 32; ++w) {
      const int t = warp_tot[w];
      if (w < warp) off += t;
      tot += t;
    }
    if (f) active[base + off + pre] = (int)c;
    __syncthreads();
    if (threadIdx.x == 0) base += tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) *n_active = base;
}

// Pooled dual averaging (B2M_ADAPT_POOLED): the recurrences of nuts.py:298-310 driven by the mean acceptance
// statistic over all chains of the call; every chain receives the same step size.  Deterministic reduction.
__global__ void __launch_bounds__(1024) nuts_pool_adapt_kernel(b2m_nuts_args A, const float *__restrict__ alpha_it, int it) {
  __shared__ double red[1024];
  __shared__ double eps_sh, hbar_sh, ebar_sh;
  const int64_t C = A.n_chains;
  double s = 0.0;
  for (int64_t c = threadIdx.x; c < C; c += 1024) {
    const float a = alpha_it[c];
    s += (a == a) ? (double)a : 0.0;
  }
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const double mean_alpha = red[0] / (double)C;
    double h_bar = A.da_state[0], eps_bar = A.da_state[1];
    const float mu = (float)A.da_state[2];
    const double m = (double)((int64_t)(uint32_t)(A.iter_offset + it) - A.adapt_origin), eta = 1.0 / (m + 10.0);
    h_bar = (1.0 - eta) * h_bar + eta * (A.target_accept - mean_alpha);
    float log_eps = __fsub_rn(mu, (float)((sqrt(m + 1.0) / 0.05) * h_bar));
    log_eps = fmaxf(fminf(log_eps, 10.0f), -10.0f);
    const double eps = (double)expf(log_eps);
    const double wgt = pow(m + 1.0, -0.75);
    eps_bar = (double)expf((float)(wgt * log(eps) + (1.0 - wgt) * log(eps_bar)));
    eps_sh = eps; hbar_sh = h_bar; ebar_sh = eps_bar;
  }
  __syncthreads();
  for (int64_t c = threadIdx.x; c < C; c += 1024) {
    A.step_size[c] = eps_sh;
    A.da_state[c * 3 + 0] = hbar_sh;
    A.da_state[c * 3 + 1] = ebar_sh;
  }
}

// carve the NUTS workspace (both schedules) out of the model's arena
static void nuts_layout(Arena &A, NutsBufs &W, int64_t C, int D, int MD) {
  const size_t cd = (size_t)C * D;
  float **vecs[] = {&W.g, &W.fq, &W.fp, &W.fg};
  for (auto v : vecs) A.take(v, cd);
  static_assert(2 * B2M_MAX_TREE_DEPTH + 2 <= 32, "the free-slot search keeps the live slots in a 32-bit mask");
  W.n_slots = 2 * MD + 2;
  A.take(&W.slots, cd * 3 * W.n_slots);
  float **fs[] = {&W.lp, &W.clp, &W.h0, &W.log_slice, &W.flp, &W.sclp, &W.feps, &W.heps};
  for (auto v : fs) A.take(v, C);
  int **is[] = {&W.n, &W.s, &W.v, &W.leaf, &W.building, &W.sub_n, &W.sub_na, &W.sub_s, &W.alpha_cnt, &W.depth,
                &W.lo, &W.hi, &W.cand, &W.leaf_slot, &W.sub_c};
  for (auto v : is) A.take(v, C);
  A.take(&W.st_f, (size_t)C * MD); A.take(&W.st_c, (size_t)C * MD);
  A.take(&W.alpha_sum, C); A.take(&W.sub_alpha, C);
  A.take(&W.st_clp, (size_t)C * MD); A.take(&W.st_n, (size_t)C * MD); A.take(&W.st_na, (size_t)C * MD);
  A.take(&W.st_alpha, (size_t)C * MD);
  A.take(&W.n_active, 1);
  A.take(&W.active, C);
  A.take(&W.alpha_it, C);
  A.take(&W.eps_it, C);
  A.take(&W.state, C); A.take(&W.iter, C); A.take(&W.fin, C); A.take(&W.live, C);
  A.take(&W.n_done, 1);
  A.take(&W.pool, 4);
}

// ================================================================= NUTS, iteration-asynchronous lock-step
// The synchronous schedule (glm_nuts_run_sync, below) advances all chains through the same iteration: a chain whose tree stops at depth 4
// waits for the one that runs to depth 10 (with thousands of chains some always do -- DESIGN.md 4.2), and the host
// synchronises once per doubling.  Here every chain is a small state machine advanced once per *tick*: consume the
// leaf that was just evaluated (tree bookkeeping; possibly close the doubling, the iteration, start the next
// iteration and its first doubling) and put the next leaf position into `fq`.  One tick = this kernel + ONE full-batch
// value+gradient; every chain has a leaf in every tick, a finished transition is followed immediately by the chain's
// next one, and the host only looks at a counter every few ticks.  Per chain the algorithm, the Philox slots and the
// arithmetic are those of the synchronous kernels (the same device functions), so a chain's draws are the same up to
// the batch-dependent rounding of the GLM contractions.
__device__ __forceinline__ void nuts_tick_dev(const b2m_nuts_args &A, const NutsBufs &W, int D, int64_t c, int lane) {
  B2M_ASSERT(c >= 0 && c < A.n_chains);
  const int st = W.state[c];
  B2M_ASSERT(st >= 0 && st <= 2);
  if (st == 2) return;
  int it = W.iter[c];
  B2M_ASSERT(it >= 0 && it < A.n_iter);
  B2M_ASSERT(W.depth[c] >= 0 && W.depth[c] <= A.max_tree_depth);
  // one call site per step of the state machine (each is a few thousand instructions once inlined)
  bool begin_transition = st == 0;
  int begin_doubling = -1;                                  // depth of the doubling to start, or -1
  if (st != 0) {
    const int j = W.depth[c];
    nuts_leaf_post_dev(A, W, D, c, lane, it, j);
    __syncwarp();
    if (!W.building[c]) {                                  // the subtree of doubling j is complete
      nuts_doubling_end_dev(A, W, D, c, lane, it, j);
      __syncwarp();
      if (W.s[c] && W.depth[c] < A.max_tree_depth) {
        begin_doubling = W.depth[c];
      } else {                                             // the transition is over
        nuts_end_dev(A, W, D, c, lane, it);
        __syncwarp();
        ++it;
        if (lane == 0) { W.iter[c] = it; W.fin[c] = 1; }
        if (it >= A.n_iter) {
          if (lane == 0) { W.state[c] = 2; W.live[c] = 0; atomicAdd(W.n_done, 1); }
          return;
        }
        begin_transition = true;
      }
    }
  }
  if (begin_transition) {
    nuts_begin_dev(A, W, D, c, lane, it);
    __syncwarp();
    begin_doubling = 0;
    if (st == 0 && lane == 0) W.state[c] = 1;
  }
  if (begin_doubling >= 0) {
    nuts_doubling_begin_dev(A, W, D, c, lane, it, begin_doubling);
    __syncwarp();
  }
  nuts_leaf_pre_dev(A, W, D, c, lane);
}

__global__ void __launch_bounds__(32 * WPB) nuts_tick_kernel(b2m_nuts_args A, NutsBufs W, int D, int64_t c_base, int64_t c_end) {
  const int lane = threadIdx.x & 31;
  const int64_t c = c_base + (int64_t)blockIdx.x * WPB + (threadIdx.x >> 5);   // this rank's chains: [c_base, c_end)
  if (c >= c_end) return;
  nuts_tick_dev(A, W, D, c, lane);
}

// ================================================================= NUTS, fused tick (fp16-encoded tcgen05 path)
// One tick of the asynchronous schedule used to be tick -> pack -> K5 -> K6 -> finish (+ a counter copy and an event):
// at the small configuration (100 x 10K, 1024 chains) launch latency was half of the tick.  The per-chain work of a
// tick now lives in ONE kernel, one warp per batch row:
//     finish (log p / gradient of the leaf evaluated by the previous tick, from K6's output)
//  -> tree bookkeeping (nuts_tick_dev: the same device functions as every other schedule)
//  -> pack (fp16 hi/lo operand rows of the next leaf position for K5)
// so a tick is state kernel -> K5 -> K6.  The last block to finish publishes {tick, finished chains} to mapped pinned
// host memory: the host throttles on it and never touches the stream inside the loop.
//
// Peer mode (observation sharding, B2M_SLICE_PEER): the rank runs this kernel for the chains it owns only.  `finish`
// first waits for the flags that say every rank has stored its gradient partial for these chains into this rank's
// window (K6's epilogue does those stores), sums the per-source slots in rank order, and `pack` writes the new rows
// into EVERY rank's window; the last block then raises this rank's "rows published" flag on every peer.
struct StateP {
  FinishP F;
  PackP P;
  const int *idx;            // batch row -> chain of a compacted batch, or nullptr
  int64_t n_rows;            // live rows [row_base, row_base + n_rows); rows up to row_base + n_pad are zero padding
  int64_t n_pad;
  int64_t row_base;          // peer mode: first chain of this rank's slice
  int do_finish, do_tick_pack;
  unsigned *blk_counter;
  volatile long long *h_prog;   // ring of {tick + 1, finished chains} pairs (non-peer mode), or nullptr
  long long tick;
  // peer mode
  int peer, nranks, rank;
  unsigned long long wait_seq, seq;
  const unsigned long long *gflag;            // [nranks] in MY window
  unsigned long long *bflag_peer[kMaxPeers];  // &bflag[rank] in every rank's window
  long long *done_peer[kMaxPeers];            // &done[rank] in every rank's window
  int *err;                                   // in my window
};

constexpr int kProgRing = 8;
constexpr long long kSpinTimeout = 20000000000ll;   // cycles (~10 s): a lost peer fails the call instead of hanging the GPU

__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long *p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long *p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// thread-level wait for *flag >= want; gives up (and records it) after kSpinTimeout cycles or when a peer already has
__device__ __forceinline__ void spin_until(const unsigned long long *flag, unsigned long long want, int *err) {
  const long long t0 = clock64();
  while (ld_acquire_sys(flag) < want) {
    if (*reinterpret_cast<volatile int *>(err)) return;
    if (clock64() - t0 > kSpinTimeout) { *reinterpret_cast<volatile int *>(err) = 1; __threadfence_system(); return; }
    __nanosleep(64);
  }
}

template <bool LIN>
__global__ void __launch_bounds__(32 * WPB, 7) nuts_state_kernel(b2m_nuts_args A, NutsBufs W, int D, KModel prior, StateP S) {
  extern __shared__ __align__(16) unsigned char smem[];
  SModel sm;
  sm.n_terms = 0;
  if (S.do_finish && S.F.has_prior) model_to_smem(prior, smem, sm);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (S.peer && S.do_finish) {   // gradient partials of the previous evaluation: one flag per source rank
    if ((int)threadIdx.x < S.nranks) spin_until(S.gflag + threadIdx.x, S.wait_seq, S.err);
    __syncthreads();
  }
  const int64_t r = (int64_t)blockIdx.x * WPB + warp;
  if (r < S.n_rows) {
    const int64_t row = S.row_base + r;
    const int64_t c = S.idx ? S.idx[row] : row;
    B2M_ASSERT(c >= 0 && c < A.n_chains && row >= 0 && (S.peer || row < S.n_pad));
    if (S.do_finish) {
      finish_row<LIN>(S.F, sm, W.fq + c * D, S.peer ? r : row, row, W.flp + c, W.fg + c * D, lane);
      __syncwarp();
    }
    if (S.do_tick_pack) {
      nuts_tick_dev(A, W, D, c, lane);
      __syncwarp();
      pack16_row(S.P, W.fq + c * D, row, lane);
    }
  } else if (r < S.n_pad && S.do_tick_pack) {
    pack16_row(S.P, nullptr, S.row_base + r, lane);
  }
  if (!S.do_tick_pack) return;
  // the last WARP to get here publishes the tick (no block-wide barrier: a warp whose chain closes a transition must
  // not hold up its three neighbours -- barrier stalls were as large as the memory stalls at 1024 chains)
  if (S.peer) __threadfence_system(); else __threadfence();
  __syncwarp();
  int last_warp = 0;
  if (lane == 0) {
    const unsigned prev = atomicAdd(S.blk_counter, 1u);
    last_warp = prev == gridDim.x * WPB - 1;
    if (last_warp) *S.blk_counter = 0;
  }
  last_warp = __shfl_sync(0xffffffffu, last_warp, 0);
  if (!last_warp) return;
  __threadfence();
  const long long n_done = *reinterpret_cast<volatile int *>(W.n_done);
  if (S.peer) {
    if (lane < S.nranks) {
      *reinterpret_cast<volatile long long *>(S.done_peer[lane]) = n_done;
      __threadfence_system();
      st_release_sys(S.bflag_peer[lane], S.seq);
    }
  } else if (lane == 0 && S.h_prog) {
    volatile long long *slot = S.h_prog + 2 * (S.tick % kProgRing);
    slot[1] = n_done;
    __threadfence_system();
    slot[0] = S.tick + 1;
  }
}

// Peer mode, after the state kernel: wait until every rank has published its rows for this evaluation, expand the row
// scalars (the residual's row scale depends on THIS rank's max |y0|), add up the finished-chain counts of the slices
// and publish {tick, finished chains of all slices} to the host.
__global__ void __launch_bounds__(256) obs_wait_kernel(const unsigned long long *bflag, int nranks, unsigned long long seq, int *err,
                                                       const float4 *__restrict__ meta, int64_t C,
                                                       const unsigned *__restrict__ y0max_bits, float x_rownorm_max, float weight,
                                                       float *__restrict__ inv_var, float *__restrict__ a_unscale,
                                                       float *__restrict__ r_scale, float *__restrict__ r_unscale,
                                                       const long long *done, volatile long long *h_prog, long long tick) {
  if ((int)threadIdx.x < nranks) spin_until(bflag + threadIdx.x, seq, err);
  __syncthreads();
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) {
    const float4 m = meta[c];
    inv_var[c] = m.x;
    a_unscale[c] = m.y;
    const float bound = (__uint_as_float(*y0max_bits) + sqrtf(m.z) * x_rownorm_max) * fabsf(m.x * weight);
    const float sr = pow2_scale(bound);
    r_scale[c] = sr;
    r_unscale[c] = 1.0f / sr;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    long long tot = 0;
    for (int s = 0; s < nranks; ++s) tot += reinterpret_cast<const volatile long long *>(done)[s];
    volatile long long *slot = h_prog + 2 * (tick % kProgRing);
    slot[1] = *reinterpret_cast<volatile int *>(err) ? -1 : tot;
    __threadfence_system();
    slot[0] = tick + 1;
  }
}

// Peer mode, after K6 (whose epilogue has stored the gradient tiles into the owners' windows): push the sum z^2
// partial of every chain into its owner's slot, then -- last block -- raise "partials stored" on every rank.
struct PeerP {
  int nranks, rank;
  int64_t own;
  float *ss_slot[kMaxPeers];                   // sum z^2 block [nranks][own] of every rank's window
  unsigned long long *gflag_peer[kMaxPeers];   // &gflag[rank] in every rank's window
};

__global__ void __launch_bounds__(256) obs_signal_kernel(const float *__restrict__ ss_part, int n_tiles, int64_t Cp, PeerP Q,
                                                         unsigned long long seq, unsigned *blk_counter) {
  // block (32 rows, 8 tile lanes): every thread adds the tiles t = y, y + 8, ... of its row (coalesced across the rows),
  // the eight partial sums are folded in fixed order -- deterministic, and eight times the loads in flight of a
  // thread-per-row loop (which was 23 us of every 630-us tick at 8 ranks)
  __shared__ float part[8][33];
  __shared__ int last_block;
  const int x = threadIdx.x & 31, y = threadIdx.x >> 5;
  const int64_t c = (int64_t)blockIdx.x * 32 + x;
  float v = 0.f;
  if (c < Cp)
    for (int t = y; t < n_tiles; t += 8) v += ss_part[(int64_t)t * Cp + c];
  part[y][x] = v;
  __syncthreads();
  if (y == 0 && c < Cp) {
    float tot = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) tot += part[i][x];
    const int owner = (int)(c / Q.own);
    Q.ss_slot[owner][(int64_t)Q.rank * Q.own + (c - (int64_t)owner * Q.own)] = tot;
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned prev = atomicAdd(blk_counter, 1u);
    last_block = prev == gridDim.x - 1;
    if (last_block) *blk_counter = 0;
  }
  __syncthreads();
  if (!last_block) return;
  __threadfence();
  if ((int)threadIdx.x < Q.nranks) st_release_sys(Q.gflag_peer[threadIdx.x], seq);
}

// Pooled dual averaging under the asynchronous schedule: acceptance statistics of the transitions that finished in
// this tick are added (fixed order) to a pool; every n_chains completed transitions -- one per chain on average -- the
// recurrences of nuts.py:298-310 advance once on the pool's mean and every chain gets the new step size for its next
// transition.  `flush` applies what is left at the end of the call.
__global__ void set_i64_kernel(long long *dst, const int *src) { *dst = (long long)*src; }

__global__ void __launch_bounds__(1024) nuts_pool_async_kernel(b2m_nuts_args A, NutsBufs W, int flush) {
  __shared__ double rs[1024];
  __shared__ int rc[1024];
  __shared__ double eps_sh, hbar_sh, ebar_sh;
  __shared__ int updated;
  const int64_t C = A.n_chains;
  double s = 0.0;
  int n = 0;
  for (int64_t c = threadIdx.x; c < C; c += 1024)
    if (W.fin[c]) {
      const float a = W.alpha_it[c];
      s += (a == a) ? (double)a : 0.0;
      ++n;
      W.fin[c] = 0;
    }
  rs[threadIdx.x] = s;
  rc[threadIdx.x] = n;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) { rs[threadIdx.x] += rs[threadIdx.x + o]; rc[threadIdx.x] += rc[threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    updated = 0;
    double sum = W.pool[0] + rs[0], cnt = W.pool[1] + (double)rc[0];
    if (cnt >= (double)C || (flush && cnt > 0.0)) {
      const double mean_alpha = sum / cnt;
      double h_bar = A.da_state[0], eps_bar = A.da_state[1];
      const float mu = (float)A.da_state[2];
      const double m = (double)((int64_t)(uint32_t)A.iter_offset - A.adapt_origin) + W.pool[2], eta = 1.0 / (m + 10.0);
      h_bar = (1.0 - eta) * h_bar + eta * (A.target_accept - mean_alpha);
      float log_eps = __fsub_rn(mu, (float)((sqrt(m + 1.0) / 0.05) * h_bar));
      log_eps = fmaxf(fminf(log_eps, 10.0f), -10.0f);
      const double eps = (double)expf(log_eps);
      const double wgt = pow(m + 1.0, -0.75);
      eps_bar = (double)expf((float)(wgt * log(eps) + (1.0 - wgt) * log(eps_bar)));
      eps_sh = eps; hbar_sh = h_bar; ebar_sh = eps_bar;
      W.pool[2] += 1.0;
      sum = 0.0; cnt = 0.0;
      updated = 1;
    }
    W.pool[0] = sum;
    W.pool[1] = cnt;
  }
  __syncthreads();
  if (updated)
    for (int64_t c = threadIdx.x; c < C; c += 1024) {
      A.step_size[c] = eps_sh;
      A.da_state[c * 3 + 0] = hbar_sh;
      A.da_state[c * 3 + 1] = ebar_sh;
    }
}

int glm_nuts_run_async(GlmModel &gm, const b2m_nuts_args &a, cudaStream_t st) {
  const int64_t C = a.n_chains;
  const int D = gm.Dtot, MD = a.max_tree_depth;
  NutsBufs W{};
  Arena probe;
  nuts_layout(probe, W, C, D, MD);
  if (int rc0 = arena_reserve(gm, probe.off)) return rc0;
  Arena real;
  real.base = gm.ws;
  nuts_layout(real, W, C, D, MD);
  W.tf = gm.tf;

  const int T = 32 * WPB;
  B2M_CHECK_CUDA(cudaMemsetAsync(W.state, 0, sizeof(int) * C, st));
  B2M_CHECK_CUDA(cudaMemsetAsync(W.iter, 0, sizeof(int) * C, st));
  B2M_CHECK_CUDA(cudaMemsetAsync(W.fin, 0, sizeof(int) * C, st));
  B2M_CHECK_CUDA(cudaMemsetAsync(W.live, 1, sizeof(int) * C, st));   // any non-zero pattern = live
  B2M_CHECK_CUDA(cudaMemsetAsync(W.n_done, 0, sizeof(int), st));
  B2M_CHECK_CUDA(cudaMemsetAsync(W.pool, 0, sizeof(double) * 4, st));
  int rc = glm_logp_grad(gm, a.theta, C, W.lp, W.g, st, true);

  constexpr int kCheck = 8;                 // ticks between recentring / tail compaction (one host sync each)
  constexpr int kRing = 4, kLag = 2;        // the finished-chain counter is read kLag ticks late, without a sync
  const bool pooled = a.adapt == B2M_ADAPT_POOLED;
  // Observation sharding with SLICED state (B2M_OBS_SLICE=1, no adaptation in the call, chains divide evenly over the
  // ranks): instead of every rank running the per-chain state machine and `finish` for all chains, rank r owns the
  // chains [r C/G, (r+1) C/G): the gradient partials are reduce-scattered, the rank finishes and advances its slice,
  // and the new leaf positions of all slices are all-gathered for the next pack / contraction.  Per-chain outputs
  // (draws, counters, depths) are written for the owned chains only; the final positions are all-gathered.
  int64_t own_base = 0, own_count = 0;
  if (gm.comm && a.adapt == B2M_ADAPT_NONE && a.slice_state == B2M_SLICE_NCCL) {
    const int nr = comm_nranks(gm.comm);
    if (nr > 1) {
      if (C % nr != 0 || C % 256 != 0) {   // the caller merges per-chain outputs by slice: never fall back silently
        set_error("slice_state: n_chains must be a multiple of 256 and of the number of ranks");
        return 1;
      }
      own_count = C / nr;
      own_base = own_count * comm_rank(gm.comm);
    }
  }
  const bool sliced = own_count > 0;
  const int64_t c_base = sliced ? own_base : 0, c_end = sliced ? own_base + own_count : C;
  const unsigned tick_grid = (unsigned)((c_end - c_base + WPB - 1) / WPB);
  long long *n_done_g = reinterpret_cast<long long *>(W.pool) + 3;   // spare slot of the pool block: global finished count
  // worst case: every transition of the slowest chain runs to the depth cap
  const int64_t max_ticks = (int64_t)a.n_iter * ((int64_t(1) << MD) + 1) + 2 * kCheck;
  cudaEvent_t ring[kRing];
  for (auto &e : ring) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
  long long *h_ring = reinterpret_cast<long long *>(gm.h_ring);   // pinned, kRing 8-byte counters
  for (int i = 0; i < kRing; ++i) h_ring[i] = 0;
  int64_t n_live = C;
  const int *idx = nullptr;
  // the host sees the counter kLag ticks late: the contractions of those surplus ticks return immediately
  if (!gm.comm) { gm.skip_flag = W.n_done; gm.skip_target = (int)C; }
  for (int64_t tick = 0; !rc; ++tick) {
    if (tick > max_ticks) { set_error("NUTS asynchronous schedule: tick budget exceeded"); rc = 2; break; }
    if (tick >= kLag) {   // the counter as it was kLag ticks ago: the device always has kLag ticks queued, the host
      cudaEventSynchronize(ring[(tick - kLag) % kRing]);   // never waits on an empty stream
      if (h_ring[(tick - kLag) % kRing] >= C) break;
    }
    nuts_tick_kernel<<<tick_grid, T, 0, st>>>(a, W, D, c_base, c_end);
    ++g_launches;
    if (sliced) {   // the counter of this rank's slice, widened and summed over ranks; then every rank's new leaf positions
      set_i64_kernel<<<1, 1, 0, st>>>(n_done_g, W.n_done);
      ++g_launches;
      if ((rc = comm_allreduce_i64(gm.comm, reinterpret_cast<int64_t *>(n_done_g), 1, st))) break;
      if ((rc = comm_allgather_inplace(gm.comm, W.fq, own_count * D, 4, st))) break;
      if (cudaMemcpyAsync(h_ring + tick % kRing, n_done_g, sizeof(long long), cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = 2;
    } else {        // low word of the (zeroed) 64-bit ring slot
      if (cudaMemcpyAsync(h_ring + tick % kRing, W.n_done, sizeof(int), cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = 2;
    }
    if (cudaEventRecord(ring[tick % kRing], st) != cudaSuccess) rc = 2;
    if (rc) { set_error("NUTS asynchronous schedule: counter copy / event record failed"); break; }
    if (pooled) {
      nuts_pool_async_kernel<<<1, 1024, 0, st>>>(a, W, 0);
      ++g_launches;
    }
    if (tick % kCheck == kCheck - 1) {
      if (cudaEventSynchronize(ring[tick % kRing]) != cudaSuccess) { rc = 2; set_error("NUTS asynchronous schedule: stream error"); break; }
      const int64_t n_done = h_ring[tick % kRing];
      if (n_done >= C) break;
      if (sliced && (rc = comm_allgather_inplace(gm.comm, a.theta, own_count * D, 4, st))) break;
      if ((rc = glm_recenter(gm, a.theta, C, st))) break;      // reference point follows the current states
      if (n_done > 0 && !sliced) {                             // the tail: evaluate only the chains still running
        nuts_compact_kernel<<<1, 1024, 0, st>>>(W.live, C, W.active, W.n_active);
        ++g_launches;
        n_live = C - n_done;
        idx = W.active;
      }
    }
    rc = glm_logp_grad(gm, W.fq, C, W.flp, W.fg, st, false, idx, n_live, own_base, own_count);
  }
  gm.skip_flag = nullptr;
  if (!rc && sliced) rc = comm_allgather_inplace(gm.comm, a.theta, own_count * D, 4, st);   // final positions everywhere
  for (auto &e : ring) cudaEventDestroy(e);
  if (!rc && pooled) {
    nuts_pool_async_kernel<<<1, 1024, 0, st>>>(a, W, 1);
    ++g_launches;
  }
  cudaError_t e = cudaStreamSynchronize(st);
  if (rc) return rc;
  B2M_CHECK_CUDA(e);
  B2M_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int glm_nuts_run_sync(GlmModel &gm, const b2m_nuts_args &a, cudaStream_t st) {
  const int64_t C = a.n_chains;
  const int D = gm.Dtot, MD = a.max_tree_depth;
  NutsBufs W{};
  Arena probe;
  nuts_layout(probe, W, C, D, MD);
  if (int rc0 = arena_reserve(gm, probe.off)) return rc0;
  Arena real;
  real.base = gm.ws;
  nuts_layout(real, W, C, D, MD);
  W.tf = gm.tf;
  int *h_flag = gm.h_flag;
  int rc = 0;

  const unsigned grid = (unsigned)((C + WPB - 1) / WPB);
  const int T = 32 * WPB;
  rc = glm_logp_grad(gm, a.theta, C, W.lp, W.g, st, true);
  for (int it = 0; it < a.n_iter && !rc; ++it) {
    if (it > 0) rc = glm_recenter(gm, a.theta, C, st);   // reference point follows the current states
    nuts_begin_kernel<<<grid, T, 0, st>>>(a, W, D, it);
    ++g_launches;
    for (int j = 0; j < MD && !rc; ++j) {
      nuts_doubling_begin_kernel<<<grid, T, 0, st>>>(a, W, D, it, j);
      nuts_compact_kernel<<<1, 1024, 0, st>>>(W.building, C, W.active, W.n_active);
      g_launches += 2;
      cudaMemcpyAsync(h_flag, W.n_active, sizeof(int), cudaMemcpyDeviceToHost, st);
      if (cudaStreamSynchronize(st) != cudaSuccess) { rc = 2; set_error("NUTS lock-step: stream error"); break; }
      const int n_act = *h_flag;
      if (n_act == 0) break;   // every chain's trajectory has ended
      // chains that stopped growing are compacted out of the batch: the two contractions of each leaf run over
      // the n_act building chains only (rounded up to the 128-row tile)
      const bool compact = n_act < C;
      for (int leaf = 0; leaf < (1 << j) && !rc; ++leaf) {
        nuts_leaf_pre_kernel<<<grid, T, 0, st>>>(a, W, D);
        rc = glm_logp_grad(gm, W.fq, C, W.flp, W.fg, st, false, compact ? W.active : nullptr, n_act);
        nuts_leaf_post_kernel<<<grid, T, 0, st>>>(a, W, D, it, j);
        g_launches += 2;
      }
      nuts_doubling_end_kernel<<<grid, T, 0, st>>>(a, W, D, it, j);
      ++g_launches;
    }
    nuts_end_kernel<<<grid, T, 0, st>>>(a, W, D, it);
    ++g_launches;
    if (a.adapt == B2M_ADAPT_POOLED) {
      nuts_pool_adapt_kernel<<<1, 1024, 0, st>>>(a, W.alpha_it, it);
      ++g_launches;
    }
  }
  cudaError_t e = cudaStreamSynchronize(st);
  if (rc) return rc;
  B2M_CHECK_CUDA(e);
  B2M_CHECK_CUDA(cudaGetLastError());
  return 0;
}

// ================================================================= NUTS, fused-tick host loop
int glm_nuts_run_fused(GlmModel &gm, const b2m_nuts_args &a, cudaStream_t st) {
  const int64_t C = a.n_chains;
  const int D = gm.Dtot, MD = a.max_tree_depth;
  const bool peer = a.slice_state == B2M_SLICE_PEER;
  PeerWindow &pw = gm.pw;
  if (peer) {
    B2M_REQUIRE(pw.nranks >= 2 && pw.C == C, "slice_state = PEER: attach a peer window for this number of chains first "
                                               "(b2m_model_peer_attach)");
    B2M_REQUIRE(a.inj_normal == nullptr && a.trace_doubling == nullptr, "slice_state = PEER: draw injection is not supported");
  }
  NutsBufs W{};
  Arena probe;
  nuts_layout(probe, W, C, D, MD);
  if (int rc0 = arena_reserve(gm, probe.off)) return rc0;
  Arena real;
  real.base = gm.ws;
  nuts_layout(real, W, C, D, MD);
  W.tf = gm.tf;
  if (!gm.blk_counter) {
    B2M_CHECK_CUDA(cudaMalloc(reinterpret_cast<void **>(&gm.blk_counter), sizeof(unsigned) * 8));
    B2M_CHECK_CUDA(cudaMemset(gm.blk_counter, 0, sizeof(unsigned) * 8));
  }
  if (!gm.h_prog) {
    long long *hp = nullptr;
    B2M_CHECK_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&hp), sizeof(long long) * 2 * kProgRing, cudaHostAllocMapped | cudaHostAllocPortable));
    gm.h_prog = hp;
  }
  volatile long long *h_prog = gm.h_prog;
  for (int i = 0; i < 2 * kProgRing; ++i) h_prog[i] = 0;

  const int T = 32 * WPB;
  B2M_CHECK_CUDA(cudaMemsetAsync(W.state, 0, sizeof(int) * C, st));
  B2M_CHECK_CUDA(cudaMemsetAsync(W.iter, 0, sizeof(int) * C, st));
  B2M_CHECK_CUDA(cudaMemsetAsync(W.fin, 0, sizeof(int) * C, st));
  B2M_CHECK_CUDA(cudaMemsetAsync(W.live, 1, sizeof(int) * C, st));   // any non-zero pattern = live
  B2M_CHECK_CUDA(cudaMemsetAsync(W.n_done, 0, sizeof(int), st));
  B2M_CHECK_CUDA(cudaMemsetAsync(W.pool, 0, sizeof(double) * 4, st));
  // log p / gradient of the starting points (observation shards: summed over ranks by NCCL, once)
  int rc = glm_logp_grad(gm, a.theta, C, W.lp, W.g, st, true);
  if (rc) return rc;

  constexpr int kCheck = 8, kLag = 2;
  const bool pooled = a.adapt == B2M_ADAPT_POOLED;
  const int64_t own = peer ? pw.own : C, own_base = peer ? pw.own * pw.rank : 0;
  const int64_t max_ticks = (int64_t)a.n_iter * ((int64_t(1) << MD) + 1) + 2 * kCheck;
  int64_t n_live = C;
  const int *idx = nullptr;
  // peer mode: K5 reads the packed rows from the window (every owner writes its rows there); restored on exit
  __half *const saved_bh = gm.B16h, *const saved_bl = gm.B16l;
  PeerP Q{};
  if (peer) {
    gm.B16h = reinterpret_cast<__half *>(pw.base[pw.rank] + pw.off_bh);
    gm.B16l = reinterpret_cast<__half *>(pw.base[pw.rank] + pw.off_bl);
    Q.nranks = pw.nranks; Q.rank = pw.rank; Q.own = pw.own;
    for (int s = 0; s < pw.nranks; ++s) {
      Q.ss_slot[s] = reinterpret_cast<float *>(pw.base[s] + pw.off_ss);
      Q.gflag_peer[s] = reinterpret_cast<unsigned long long *>(pw.base[s] + pw.off_gflag) + pw.rank;
    }
  } else if (!gm.comm) {
    gm.skip_flag = W.n_done;   // the contractions of the ticks the host launches after the last chain finished return at once
    gm.skip_target = (int)C;
  }
  auto cleanup = [&]() { gm.B16h = saved_bh; gm.B16l = saved_bl; gm.skip_flag = nullptr; };

  auto state_params = [&](bool do_finish, bool do_tick_pack, int64_t tick, unsigned long long wait_seq, unsigned long long seq) {
    StateP S{};
    const int64_t rows = idx ? n_live : C;
    const int64_t Cp = rows <= 128 ? 128 : (rows + 255) / 256 * 256;
    S.F = make_finish(gm, peer ? own : Cp, true);
    S.P = make_pack(gm);
    S.idx = idx;
    S.n_rows = peer ? own : rows;
    S.n_pad = peer ? own : Cp;
    S.row_base = own_base;
    S.do_finish = do_finish ? 1 : 0;
    S.do_tick_pack = do_tick_pack ? 1 : 0;
    S.blk_counter = gm.blk_counter;
    S.h_prog = peer ? nullptr : h_prog;
    S.tick = tick;
    S.peer = peer ? 1 : 0;
    if (peer) {
      S.nranks = pw.nranks; S.rank = pw.rank;
      S.wait_seq = wait_seq; S.seq = seq;
      char *mine = pw.base[pw.rank];
      S.gflag = reinterpret_cast<const unsigned long long *>(mine + pw.off_gflag);
      S.err = reinterpret_cast<int *>(mine + pw.off_err);
      // finish: per-source slots of my window, summed in rank order; already unscaled by the senders
      S.F.G = reinterpret_cast<const float *>(mine + pw.off_g);
      S.F.ss_part = reinterpret_cast<const float *>(mine + pw.off_ss);
      S.F.g_splits = pw.nranks; S.F.n_tiles = pw.nranks; S.F.Cp = own;
      S.F.r_unscale = nullptr; S.F.inv_col_scale = nullptr;
      S.P.n_peers = pw.nranks;
      for (int s = 0; s < pw.nranks; ++s) {
        S.P.peer_Bh[s] = reinterpret_cast<__half *>(pw.base[s] + pw.off_bh);
        S.P.peer_Bl[s] = reinterpret_cast<__half *>(pw.base[s] + pw.off_bl);
        S.P.peer_meta[s] = reinterpret_cast<float4 *>(pw.base[s] + pw.off_meta);
        S.bflag_peer[s] = reinterpret_cast<unsigned long long *>(pw.base[s] + pw.off_bflag) + pw.rank;
        S.done_peer[s] = reinterpret_cast<long long *>(pw.base[s] + pw.off_done) + pw.rank;
      }
    }
    return S;
  };
  auto launch_state = [&](const StateP &S) {
    const unsigned grid = (unsigned)((S.n_pad + WPB - 1) / WPB);
    prof_mark(2, st);
    (gm.prior_lin ? nuts_state_kernel<true> : nuts_state_kernel<false>)<<<grid, T, finish_smem(gm), st>>>(a, W, D, gm.prior, S);
    prof_mark(2, st);
    ++g_launches;
  };
  // host side of the progress ring: {tick + 1, finished chains} of tick t lives in slot t % kProgRing
  auto wait_tick = [&](int64_t t, long long &n_done) -> int {
    volatile long long *slot = h_prog + 2 * (t % kProgRing);
    const auto t0 = std::chrono::steady_clock::now();
    for (unsigned spins = 0; slot[0] != t + 1; ++spins) {
      if ((spins & 0xfff) == 0xfff) {
        if (cudaStreamQuery(st) != cudaErrorNotReady && slot[0] != t + 1) {   // the stream drained (or failed) without the tick
          set_error("NUTS fused schedule: the device stopped before publishing a tick");
          return 2;
        }
        if (std::chrono::steady_clock::now() - t0 > std::chrono::seconds(120)) {
          set_error("NUTS fused schedule: timed out waiting for the device");
          return 2;
        }
      }
    }
    n_done = slot[1];
    if (n_done < 0) { set_error("NUTS peer exchange: a rank stopped answering (flag wait timed out)"); return 2; }
    return 0;
  };

  unsigned long long prev_seq = 0;
  for (int64_t tick = 0; !rc; ++tick) {
    if (tick > max_ticks) { set_error("NUTS fused schedule: tick budget exceeded"); rc = 2; break; }
    const bool check = tick > 0 && tick % kCheck == 0;
    long long n_done = 0;
    if (check) {
      // finish the leaf of tick - 1 with the row mapping it was evaluated under, then drain: recentre / compact
      launch_state(state_params(true, false, tick, prev_seq, 0));
      if ((rc = wait_tick(tick - 1, n_done))) break;
      if (n_done >= C) break;
      if (peer && (rc = comm_allgather_inplace(gm.comm, a.theta, own * D, 4, st))) break;
      if ((rc = glm_recenter(gm, a.theta, C, st))) break;      // reference point follows the current states
      if (n_done > 0 && !peer) {                               // the tail: evaluate only the chains still running
        nuts_compact_kernel<<<1, 1024, 0, st>>>(W.live, C, W.active, W.n_active);
        ++g_launches;
        n_live = C - n_done;
        idx = W.active;
      }
    } else if (tick >= kLag) {   // the device always has kLag ticks queued; the host never drains the stream
      if ((rc = wait_tick(tick - kLag, n_done))) break;
      if (n_done >= C) break;
    }
    const unsigned long long seq = peer ? ++pw.seq : 0;
    launch_state(state_params(tick > 0 && !check, true, tick, prev_seq, seq));
    prev_seq = seq;
    if (pooled) {
      nuts_pool_async_kernel<<<1, 1024, 0, st>>>(a, W, 0);
      ++g_launches;
    }
    const int64_t rows = idx ? n_live : C;
    const int64_t Cp = rows <= 128 ? 128 : (rows + 255) / 256 * 256;
    if (peer) {
      char *mine = pw.base[pw.rank];
      prof_mark(3, st);
      obs_wait_kernel<<<(unsigned)((C + 255) / 256), 256, 0, st>>>(
          reinterpret_cast<const unsigned long long *>(mine + pw.off_bflag), pw.nranks, seq,
          reinterpret_cast<int *>(mine + pw.off_err), reinterpret_cast<const float4 *>(mine + pw.off_meta), C, gm.y0max_bits,
          gm.x_rownorm_max, gm.weight, gm.inv_var, gm.a_unscale, gm.r_scale, gm.r_unscale,
          reinterpret_cast<const long long *>(mine + pw.off_done), h_prog, tick);
      prof_mark(3, st);
      ++g_launches;
    }
    if (gm.form == kFormGram) {   // one contraction against the Gram operand (never sharded)
      if ((rc = tc_gemm_gram(gm, Cp, st))) break;
    } else if (!peer) {
      if ((rc = tc_gemm_resid(gm, Cp, st))) break;
      if ((rc = tc_gemm_grad(gm, Cp, st))) break;
    } else {
      if ((rc = tc_gemm_resid(gm, Cp, st))) break;
      if ((rc = tc_gemm_grad_push(gm, Cp, st))) break;
      prof_mark(4, st);
      obs_signal_kernel<<<(unsigned)((Cp + 31) / 32), 256, 0, st>>>(gm.ss_part, gm.Np / 128, Cp, Q, seq, gm.blk_counter + 1);
      prof_mark(4, st);
      ++g_launches;
    }
    if (cudaGetLastError() != cudaSuccess) { set_error("NUTS fused schedule: launch failed"); rc = 2; }
  }
  cleanup();
  if (!rc && peer) rc = comm_allgather_inplace(gm.comm, a.theta, own * D, 4, st);   // final positions everywhere
  if (!rc && pooled) {
    nuts_pool_async_kernel<<<1, 1024, 0, st>>>(a, W, 1);
    ++g_launches;
  }
  cudaError_t e = cudaStreamSynchronize(st);
  if (rc) return rc;
  B2M_CHECK_CUDA(e);
  B2M_CHECK_CUDA(cudaGetLastError());
  if (peer) {
    int herr = 0;
    B2M_CHECK_CUDA(cudaMemcpy(&herr, pw.base[pw.rank] + pw.off_err, sizeof(int), cudaMemcpyDeviceToHost));
    B2M_REQUIRE(herr == 0, "NUTS peer exchange: a flag wait timed out");
  }
  return 0;
}

// schedule / slicing come with the call (b2m_nuts_args; environment variables in ABI 1).  The fused tick needs the
// fp16-encoded tensor-core path and no draw injection bookkeeping beyond what the device functions already do; the
// NCCL forms of observation sharding (replicated state, or reduce-scatter + all-gather slicing) keep the unfused loop.
int glm_nuts_run(GlmModel &gm, const b2m_nuts_args &a, cudaStream_t st) {
  if (a.schedule == B2M_SCHED_SYNC) return glm_nuts_run_sync(gm, a, st);
  const bool fused_ok = gm.use_tc == 2 && (!gm.comm || a.slice_state == B2M_SLICE_PEER);
  if (a.slice_state == B2M_SLICE_PEER && !fused_ok) {
    set_error("slice_state = PEER needs the fp16-encoded tensor-core path");
    return 1;
  }
  if (fused_ok) return glm_nuts_run_fused(gm, a, st);
  return glm_nuts_run_async(gm, a, st);
}

}  // namespace b2m

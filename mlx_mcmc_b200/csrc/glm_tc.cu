// K5 / K6 on the 5th-generation tensor cores: TMA-staged tcgen05 GEMMs in 3xTF32.
//
//   D[m, n] = sum_k (Ah + Al)[m, k] * (Bh + Bl)[n, k]   ~=   Ah.Bh + Ah.Bl + Al.Bh      (fp32 accumulate in TMEM)
//
// Every operand is K-major fp32 holding tf32-representable values (round-to-nearest hi/lo split, glm.cuh), so
// the dropped Al.Bl term is ~2^-22 relative: the two contractions hold the 1e-5 log-prob / gradient tolerance.
//
// Two launch shapes share the kernel body (template NCTA):
//   NCTA = 1   one CTA = one 128 x BLOCK_N tile                                   (small / compacted batches)
//   NCTA = 2   a CTA pair (cluster of 2, tcgen05 cta_group::2) = one 256 x BLOCK_N tile: each CTA stages its own
//              128 rows of A and HALF of the B tile, the leader CTA issues the MMAs for both, each CTA's TMEM
//              receives its own 128 rows.  Per k-block a CTA pulls 64 KB instead of 96 KB through L2 -- the v1
//              kernel was pinned at the ~6300 B/clk L2->SM return path (profiles/r01_tc_gemm_c4_v1_ncu_summary.md).
//
// Kernel anatomy (one 128 x BLOCK_N output tile per CTA, 320 threads):
//   warp 0      TMA producer: cp.async.bulk.tensor 2-D loads of the four operand tiles of a k-block
//               (BLOCK_K = 32 floats = one 128-byte swizzle row) into a ring of shared-memory stages
//   warp 1      TMEM allocator + single-thread tcgen05.mma issuer (3 MMAs x 4 k-steps per stage),
//               tcgen05.commit releases the stage / hands a finished K-chunk to the promotion warps
//   warps 2..9  promotion + epilogue.  The tensor core adds into its fp32 accumulator with truncation, so a
//               long K loop drifts (~T * 2^-24 relative after T MMAs: measured 4e-6 at K = 1000, would be
//               ~2e-3 at K = 100,000).  Therefore TMEM holds only a CHUNK of 4 k-blocks (K = 128) at a time,
//               double buffered; these warps tcgen05.ld each finished chunk and add it round-to-nearest into
//               fp32 master accumulators in registers (lane = output row, 8 warps = 4 lane quarters x 2 column
//               halves).  At the end:
//                 RESID: z = y - c - acc, per-row sum z^2, R = w z / sigma^2 split into tf32 hi/lo   (K5)
//                 LOGIT: eta = eta0 + acc, per-row sum of y eta - softplus(eta), R = w (y - sigmoid(eta))
//                        (K5 of the Bernoulli-logit likelihood, same transposition and stores as RESID)
//                 PLAIN: store the split-K partial of G                                              (K6)
//                 STATS: per element the pointwise log-likelihood ll of the Normal or Bernoulli-logit kind, reduced
//                        over the warp's 32 chain rows per observation into (max, sum exp(ll - max), mean, M2)
//                        partials (b2m_loglik_stats: K5 over posterior draws instead of chains, no R written)
#include <cuda.h>
#include <cuda_fp16.h>

#include <atomic>
#include <vector>

#include "glm.cuh"

namespace b2m {

namespace {

constexpr int BLOCK_M = 128;
constexpr int ROW_BYTES = 128;                        // one SWIZZLE_128B row of K: 32 tf32 values or 64 fp16 values
constexpr int MMA_K_BYTES = 32;                       // one MMA k-step: 8 tf32 or 16 fp16 values
constexpr int A_TILE_BYTES = BLOCK_M * ROW_BYTES;     // 16 KB
// elements of K per k-block (one swizzle row) for the two operand encodings
template <bool F16> struct Enc { static constexpr int BLOCK_K = F16 ? 64 : 32; };
constexpr int BLOCK_K = 32;                           // tf32 k-block (host-side helpers of the tf32 path)
constexpr int NUM_EPI_WARPS = 8;
constexpr int NUM_THREADS = 64 + 32 * NUM_EPI_WARPS;   // TMA warp, MMA warp, 8 promotion/epilogue warps
constexpr int DEFAULT_CHUNK_KB = 4;                     // k-blocks accumulated inside the tensor core per chunk

// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done;
  do {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
  } while (!done);
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// ---- cluster / CTA-pair helpers
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `local` (a shared::cta address) inside CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa(uint32_t local, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  // default semantics (release at CTA scope), as CUTLASS's ClusterBarrier::arrive(cta_id): the arrival only says "this
  // warp has drained its TMEM reads / issued its loads"; a cluster-scope release compiled to MEMBAR.ALL.GPU + ERRBAR
  // and was 7 % of the K5 stall samples
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA load issued by one CTA of a pair; completion bytes are signalled on the LEADER's mbarrier (cluster address)
__device__ __forceinline__ void tma_load_2d_pair(void *dst, const CUtensorMap *map, uint32_t leader_bar, int x, int y) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(leader_bar), "r"(x), "r"(y)
      : "memory");
}
__device__ __forceinline__ void umma_tf32_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// commit of the pair's MMAs: arrives on the mbarrier at the same offset in BOTH CTAs
__device__ __forceinline__ void umma_commit_pair(uint64_t *bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"((uint16_t)3)
               : "memory");
}

__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, uint64_t *bar, int x, int y) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(x), "r"(y)
      : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
template <bool F16, int NCTA>
__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  if (F16) {
    if (NCTA == 2) umma_f16_pair(tmem_d, adesc, bdesc, idesc, accumulate); else umma_f16(tmem_d, adesc, bdesc, idesc, accumulate);
  } else {
    if (NCTA == 2) umma_tf32_pair(tmem_d, adesc, bdesc, idesc, accumulate); else umma_tf32(tmem_d, adesc, bdesc, idesc, accumulate);
  }
}
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor layout):
// start address >> 4 | LBO (unused for swizzled K-major, = 1) << 16 | SBO = 1024 B (8 rows x 128 B) >> 4 << 32 |
// version 1 << 46 | layout SWIZZLE_128B (2) << 61
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) |
         ((uint64_t)2 << 61);
}

// instruction descriptor (cute::UMMA::InstrDescriptor): D = F32, A = B = TF32, both K-major, N >> 3, M >> 4
// a_format / b_format: 0 = F16, 2 = TF32
__host__ __device__ constexpr uint32_t make_idesc(int n, int m = BLOCK_M, bool f16 = false) {
  return (1u << 4) | ((f16 ? 0u : 2u) << 7) | ((f16 ? 0u : 2u) << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

struct EpiParams {
  // RESID
  const float *y;
  const float *inv_var;
  void *Rh, *Rl;          // [Cp, Np] residual operand of K6: float (tf32 values) or __half
  float *ss_part;
  const float *a_unscale; // F16: [Cp] 1 / (row scale of the A operand), applied to the accumulators
  const float *r_scale;   // F16: [Cp] row scale of R before the fp16 split
  int64_t Cp;
  int Np, N_valid;
  float loc_const, weight;
  // PLAIN
  float *Gpart;  // [splits, Cp, Dp]
  int Dp;
  // both: the launch is a no-op once *skip_flag >= skip_target (every chain of the call has finished; the host learns
  // it a few launches late because it reads the counter without draining the stream)
  const int *skip_flag;
  int skip_target;
  // PUSH (K6 of a peer-sliced observation shard): the finished tile goes, unscaled, straight into the window of the
  // rank that owns its chains -- slot `push_rank` of that rank's [nranks][own][Dp] gradient block -- over NVLink
  float *push_dst[kMaxPeers];
  int push_own, push_rank;
  const float *r_unscale;       // [Cp]
  const float *inv_col_scale;   // [Dp]
  // LOGIT (last, so that the parameter offsets of the other modes stay where they were)
  const float *eta0;      // [Np] c + X beta0 (float64-accumulated centring, padding -inf); `y` holds the labels
  // STATS: [Cp / 32, Np] partials of 32 draw rows each; rows >= rows_valid of the batch are excluded
  float4 *part;
  int64_t rows_valid;
};

template <int BLOCK_N, int NCTA>
struct Cfg {
  static constexpr int B_ROWS = BLOCK_N / NCTA;         // rows of the B tile staged by one CTA
  static constexpr int B_TILE_BYTES = B_ROWS * ROW_BYTES;
  static constexpr int STAGE_BYTES = 2 * A_TILE_BYTES + 2 * B_TILE_BYTES;
  static constexpr int STAGES = (192 * 1024) / STAGE_BYTES > 6 ? 6 : (192 * 1024) / STAGE_BYTES;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*alignment slack*/ + 256 /*barriers*/;
  static constexpr int TMEM_COLS = 2 * BLOCK_N;        // two chunk accumulators (power of two >= 32)
  static constexpr int COLS_PER_WARP = BLOCK_N / 2;    // each promotion warp owns 32 rows x half of the columns
};

// MODE: 0 = PLAIN (split-K partial of G), 1 = RESID (K5 residual epilogue), 2 = PUSH (K6 tile -> owner's window),
//       3 = LOGIT (K5 with the Bernoulli-logit residual epilogue), 4 / 5 = STATS (K5 with the log-likelihood statistics
//       epilogue, Normal / Bernoulli-logit)
template <int BLOCK_N, int MODE, int NCTA, bool F16>
__global__ void __launch_bounds__(NUM_THREADS, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap tmAh, const __grid_constant__ CUtensorMap tmAl,
               const __grid_constant__ CUtensorMap tmBh, const __grid_constant__ CUtensorMap tmBl, int k_blocks_total,
               int k_blocks_per_split, int CHUNK_KB, int mma_mask, int Tm, int Tn, int n_tiles, const __grid_constant__ EpiParams E) {
  if (E.skip_flag && *reinterpret_cast<const volatile int *>(E.skip_flag) >= E.skip_target) return;   // uniform over the grid
  using C = Cfg<BLOCK_N, NCTA>;
  constexpr bool LOGIT = MODE == 3, RESID = MODE == 1 || LOGIT, PUSH = MODE == 2;
  constexpr bool STATS = MODE == 4 || MODE == 5, STATS_LOGIT = MODE == 5;
  constexpr bool K5 = RESID || STATS;          // the B X^T tile order
  constexpr int BLOCK_K = Enc<F16>::BLOCK_K;   // K elements per k-block (shadows the tf32 constant)
  constexpr int SCRATCH_BYTES = (RESID || PUSH || STATS) ? NUM_EPI_WARPS * 32 * 33 * 4 : 0;   // per-warp transpose scratch of the epilogue
  extern __shared__ unsigned char smem_raw[];
  unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  float *scratch_base = reinterpret_cast<float *>(smem + C::STAGES * C::STAGE_BYTES);
  uint64_t *full = reinterpret_cast<uint64_t *>(smem + C::STAGES * C::STAGE_BYTES + SCRATCH_BYTES);
  uint64_t *empty = full + C::STAGES;
  uint64_t *tmem_full = empty + C::STAGES;   // [2]
  uint64_t *tmem_empty = tmem_full + 2;      // [2]
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t cta = NCTA == 2 ? cluster_ctarank() : 0u;   // rank inside the CTA pair; 0 = leader (issues the MMAs)
  const int group = (int)blockIdx.x / NCTA, n_groups = (int)gridDim.x / NCTA;
  // Persistent tile loop: CTA group g (a CTA, or a pair) takes tiles g, g + G, g + 2G, ...  K5: tile t = (pair-row
  // t % Tm, observation tile t / Tm) -- the sixteen pairs on one observation tile share the B tile (design matrix rows),
  // the A operand (packed positions, 16 MB) lives in L2.  K6: tile t = (column tile t % Tn, pair-row (t / Tn) % Tm, K split
  // t / (Tm Tn)) -- the Tn neighbours share the A tile, which is the big stream there (the residual operand: 1.6 GB per
  // evaluation at C4 against 0.4 GB of transposed design matrix); with the pair row fastest the Tn readers of one residual
  // tile were 16 tiles apart, often in different rounds of the 74 pairs, and the tile came from DRAM more than once.  Barriers and TMEM
  // are set up once; the producer and the MMA issuer run ahead into the next tile while the promotion warps are
  // still in the epilogue of the previous one (both TMEM chunk buffers are free by then).
#define B2M_DECODE_TILE(t)                                                         \
  const int mp_ = K5 ? (t) % Tm : ((t) / Tn) % Tm;                                 \
  const int nt = K5 ? ((t) / Tm) % Tn : (t) % Tn;                                  \
  const int zs = (t) / (Tm * Tn);                                                  \
  const int m0 = (mp_ * NCTA + (int)cta) * BLOCK_M, n0 = nt * BLOCK_N;             \
  const int kb0 = zs * k_blocks_per_split;                                         \
  const int kb1 = min(kb0 + k_blocks_per_split, k_blocks_total);                   \
  const int nkb = kb1 - kb0;                                                       \
  const int n_chunks = (nkb + CHUNK_KB - 1) / CHUNK_KB;                            \
  (void)m0; (void)n0; (void)nt; (void)zs; (void)nkb; (void)n_chunks;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmAh) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmAl) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmBh) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmBl) : "memory");
    // pair: the leader's `full` collects one arrival per producer (2) and the bytes of both CTAs' loads; the leader's
    // `tmem_empty` collects the promotion threads of both CTAs; `empty` / `tmem_full` are signalled in both CTAs by
    // the multicast tcgen05.commit
    for (int s = 0; s < C::STAGES; ++s) { mbar_init(&full[s], NCTA); mbar_init(&empty[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&tmem_full[b], 1); mbar_init(&tmem_empty[b], NCTA * NUM_EPI_WARPS); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    if (NCTA == 2) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(C::TMEM_COLS));
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(C::TMEM_COLS));
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  if (NCTA == 2) cluster_sync_all(); else __syncthreads();   // barriers initialised and TMEM allocated in both CTAs
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = group; t < n_tiles; t += n_groups) {
      B2M_DECODE_TILE(t)
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(&empty[stage], phase ^ 1);
        unsigned char *st = smem + stage * C::STAGE_BYTES;
        if (NCTA == 2) {
          const uint32_t lbar = mapa(smem_u32(&full[stage]), 0);   // the leader's barrier
          if (cta == 0) mbar_expect_tx(&full[stage], 2 * C::STAGE_BYTES);
          else mbar_arrive_cluster(lbar);
          const int nb = n0 + (int)cta * C::B_ROWS;               // this CTA's half of the B tile
          tma_load_2d_pair(st, &tmAh, lbar, kb * BLOCK_K, m0);
          tma_load_2d_pair(st + A_TILE_BYTES, &tmAl, lbar, kb * BLOCK_K, m0);
          tma_load_2d_pair(st + 2 * A_TILE_BYTES, &tmBh, lbar, kb * BLOCK_K, nb);
          tma_load_2d_pair(st + 2 * A_TILE_BYTES + C::B_TILE_BYTES, &tmBl, lbar, kb * BLOCK_K, nb);
        } else {
          mbar_expect_tx(&full[stage], C::STAGE_BYTES);
          tma_load_2d(st, &tmAh, &full[stage], kb * BLOCK_K, m0);
          tma_load_2d(st + A_TILE_BYTES, &tmAl, &full[stage], kb * BLOCK_K, m0);
          tma_load_2d(st + 2 * A_TILE_BYTES, &tmBh, &full[stage], kb * BLOCK_K, n0);
          tma_load_2d(st + 2 * A_TILE_BYTES + C::B_TILE_BYTES, &tmBl, &full[stage], kb * BLOCK_K, n0);
        }
        if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
      }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (one elected lane) =====
    if (lane == 0 && cta == 0) {
      constexpr uint32_t idesc = make_idesc(BLOCK_N, BLOCK_M * NCTA, F16);
      int stage = 0;
      uint32_t phase = 0;
      uint32_t gch = 0;   // chunk counter across tiles: buffer = gch & 1, barrier parity = (gch >> 1) & 1
      for (int t = group; t < n_tiles; t += n_groups) {
      B2M_DECODE_TILE(t)
      int kb = 0;
      for (int ch = 0; ch < n_chunks; ++ch, ++gch) {
        const int buf = gch & 1;
        mbar_wait(&tmem_empty[buf], ((gch >> 1) & 1) ^ 1);   // the promotion warps have drained this buffer
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t tmem_d = tmem_base + buf * BLOCK_N;
        const int kb_end = min(kb + CHUNK_KB, nkb);
        for (int kc = 0; kb < kb_end; ++kb, ++kc) {
          mbar_wait(&full[stage], phase);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t st = smem_u32(smem + stage * C::STAGE_BYTES);
          const uint64_t dAh = make_desc(st), dAl = make_desc(st + A_TILE_BYTES);
          const uint64_t dBh = make_desc(st + 2 * A_TILE_BYTES), dBl = make_desc(st + 2 * A_TILE_BYTES + C::B_TILE_BYTES);
#pragma unroll
          for (int k = 0; k < ROW_BYTES / MMA_K_BYTES; ++k) {
            const uint64_t adv = (uint64_t)((k * MMA_K_BYTES) >> 4);  // start-address advance inside the swizzle row
            umma<F16, NCTA>(tmem_d, dAh + adv, dBh + adv, idesc, (kc | k) != 0 ? 1u : 0u);
            if (mma_mask & 2) umma<F16, NCTA>(tmem_d, dAh + adv, dBl + adv, idesc, 1u);
            if (mma_mask & 4) umma<F16, NCTA>(tmem_d, dAl + adv, dBh + adv, idesc, 1u);
          }
          // frees the stage (in both CTAs of a pair) once the MMAs above have read it
          if (NCTA == 2) umma_commit_pair(&empty[stage]); else umma_commit(&empty[stage]);
          if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
        }
        // chunk accumulator complete (in both CTAs' TMEM)
        if (NCTA == 2) umma_commit_pair(&tmem_full[buf]); else umma_commit(&tmem_full[buf]);
      }
      }
    }
  } else {
    // ===== promotion + epilogue warps: TMEM lane quarter = warp % 4, column half = (warp - 2) / 4 =====
    const int q = warp & 3, half = (warp - 2) >> 2;
    constexpr int CW = C::COLS_PER_WARP;
    uint32_t gch = 0;
    for (int t = group; t < n_tiles; t += n_groups) {
    B2M_DECODE_TILE(t)
    const int m = m0 + q * 32 + lane;
    B2M_ASSERT(m >= 0 && (int64_t)m < E.Cp && nkb > 0);
    float acc[CW];
#pragma unroll
    for (int j = 0; j < CW; ++j) acc[j] = 0.f;
    for (int ch = 0; ch < n_chunks; ++ch, ++gch) {
      const int buf = gch & 1;
      mbar_wait(&tmem_full[buf], (gch >> 1) & 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16) + buf * BLOCK_N + half * CW;
#pragma unroll
      for (int cb = 0; cb < CW / 32; ++cb) {
        uint32_t v[32];
        tmem_ld32(trow + cb * 32, v);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[cb * 32 + j] += __uint_as_float(v[j]);   // round-to-nearest promotion
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) {   // one arrival per warp: a cluster-scope release per thread was 13 % of the v2 stall samples
        if (NCTA == 2) mbar_arrive_cluster(mapa(smem_u32(&tmem_empty[buf]), 0));   // the leader's MMA warp waits on it
        else mbar_arrive(&tmem_empty[buf]);
      }
    }
    const int nb = n0 + half * CW;
    if (RESID) {
      // Residual epilogue.  The thread owns row m (a chain) and CW consecutive columns (observations); written
      // straight from registers each store instruction would touch 32 different rows (16 B per row: uncoalesced,
      // partial-sector writes -- the first version spent more time here than in the MMAs).  Each warp therefore
      // transposes 32x32 blocks through a private shared-memory scratch (33-float pitch: conflict-free both ways)
      // and stores whole 128-byte row segments.
      float ss = 0.f;   // Normal: sum z^2; LOGIT: sum of the Bernoulli log-likelihood terms
      const float ivw = LOGIT ? E.weight : E.inv_var[m] * E.weight;
      // F16: the accumulators carry the row scale of the A operand (delta); R gets its own row scale before the split
      const float a_un = F16 ? E.a_unscale[m] : 1.0f;
      const float rs_lane = F16 ? E.r_scale[m] : 1.0f;   // lane r holds the R scale of row r of this warp's 32 rows
      float *scratch = scratch_base + (warp - 2) * (32 * 33);
      const int64_t row0 = (int64_t)(m0 + q * 32);
      // the observations of this warp's columns: one coalesced load per 32-column block (lane = column), handed to
      // the row-owning threads by shuffle (a per-element __ldg serialised 128 L2 round trips per thread)
      float yv[CW / 32], ev[LOGIT ? CW / 32 : 1];
#pragma unroll
      for (int b = 0; b < CW / 32; ++b) {
        const int n = nb + b * 32 + lane;
        if (LOGIT) {   // labels and eta0: both arrays are Np long, the padding needs no test (eta0 = -inf there)
          yv[b] = __ldg(E.y + n);
          ev[b] = __ldg(E.eta0 + n);
        } else {
          yv[b] = (n < E.N_valid) ? __ldg(E.y + n) - E.loc_const : 0.f;
        }
      }
      // (columns n >= N_valid need no test below: the padded rows of X are zero, so acc = 0 there, and yv = 0; LOGIT:
      // label 0 and eta = -inf give a zero term and a zero residual)
#pragma unroll
      for (int b = 0; b < CW / 32; ++b) {
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float yj = __shfl_sync(0xffffffffu, yv[b], j);
          const float xd = F16 ? acc[b * 32 + j] * a_un : acc[b * 32 + j];
          float r;
          if (LOGIT) {
            // one exp(-|eta|) feeds softplus and sigmoid (bernoulli_logit, model.cuh)
            float lp, dt;
            bernoulli_logit(yj != 0.f, __shfl_sync(0xffffffffu, ev[b], j) + xd, lp, dt);
            ss += lp;
            r = dt * ivw;
          } else {
            const float z = yj - xd;
            ss = fmaf(z, z, ss);
            r = z * ivw;
          }
          // F16: the row scale of R is applied here, by the thread that owns the row (same two multiplications, in the
          // same order, as scaling after the transposition -- without a shuffle and two multiplies per stored pair)
          scratch[lane * 33 + j] = F16 ? r * rs_lane : r;
        }
        __syncwarp();
        if (F16) {
          // two rows per instruction: lanes 0-15 take row r, lanes 16-31 row r + 1, each lane two adjacent columns
          // (bank = 33 row + 2 col': even banks for one half-warp, odd for the other -- conflict free) packed into
          // one half2 store per array: half the conversions and half the store instructions of a per-element loop
          const int hrow = lane >> 4, cl = (lane & 15) * 2;
          const int64_t off = (row0 + hrow) * E.Np + nb + b * 32 + cl;
          __half2 *rh = reinterpret_cast<__half2 *>(static_cast<__half *>(E.Rh) + off);
          __half2 *rl = reinterpret_cast<__half2 *>(static_cast<__half *>(E.Rl) + off);
#pragma unroll 8
          for (int r = 0; r < 32; r += 2) {
            const float v0 = scratch[(r + hrow) * 33 + cl], v1 = scratch[(r + hrow) * 33 + cl + 1];
            const __half2 hi = __floats2half2_rn(v0, v1);
            const float2 hf = __half22float2(hi);
            rh[(int64_t)r * (E.Np / 2)] = hi;
            rl[(int64_t)r * (E.Np / 2)] = __floats2half2_rn(v0 - hf.x, v1 - hf.y);
          }
        } else {
          const int64_t off = row0 * E.Np + nb + b * 32 + lane;
          float *rh = static_cast<float *>(E.Rh) + off, *rl = static_cast<float *>(E.Rl) + off;
#pragma unroll 8
          for (int r = 0; r < 32; ++r) {
            float hi, lo;
            split_tf32(scratch[r * 33 + lane], hi, lo);
            rh[(int64_t)r * E.Np] = hi;
            rl[(int64_t)r * E.Np] = lo;
          }
        }
        __syncwarp();
      }
      E.ss_part[((int64_t)nt * 2 + half) * E.Cp + m] = ss;
    } else if (STATS) {
      // Statistics epilogue.  The thread that owns row m (a draw) computes ll for its CW columns and transposes each
      // 32 x 32 block through the warp's scratch, as the residual epilogue does; afterwards lane l owns observation
      // nb + 32 b + l over the warp's 32 rows and reduces that column: max and sum exp(ll - max), then the mean and, in
      // a second pass, M2 = sum (ll - mean)^2 (fp32 sum ll^2 - (sum ll)^2 / n cancels where the variance is small).
      const float a_un = F16 ? E.a_unscale[m] : 1.0f;
      const float iv = STATS_LOGIT ? 1.0f : E.inv_var[m];
      const float lbase = STATS_LOGIT ? 0.f : 0.5f * logf(iv) - kHalfLog2Pi;
      float *scratch = scratch_base + (warp - 2) * (32 * 33);
      const int64_t row0 = (int64_t)(m0 + q * 32);
      const int64_t left = E.rows_valid - row0;
      const int nv = left >= 32 ? 32 : (left > 0 ? (int)left : 0);   // draw rows of this warp that count (uniform)
      float yv[CW / 32], ev[STATS_LOGIT ? CW / 32 : 1];
#pragma unroll
      for (int b = 0; b < CW / 32; ++b) {
        const int n = nb + b * 32 + lane;
        if (STATS_LOGIT) {
          yv[b] = __ldg(E.y + n);
          ev[b] = __ldg(E.eta0 + n);
        } else {
          yv[b] = (n < E.N_valid) ? __ldg(E.y + n) : 0.f;
        }
      }
#pragma unroll
      for (int b = 0; b < CW / 32; ++b) {
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float yj = __shfl_sync(0xffffffffu, yv[b], j);
          const float xd = F16 ? acc[b * 32 + j] * a_un : acc[b * 32 + j];
          float ll;
          if (STATS_LOGIT) {
            float dt;
            bernoulli_logit(yj != 0.f, __shfl_sync(0xffffffffu, ev[b], j) + xd, ll, dt);
          } else {
            const float z = yj - xd;
            ll = lbase - 0.5f * (iv * (z * z));
          }
          scratch[lane * 33 + j] = ll * E.weight;
        }
        __syncwarp();
        const int n = nb + b * 32 + lane;
        if (nv > 0 && n < E.N_valid) {
          float mx = -INFINITY, s = 0.f;
          for (int r = 0; r < nv; ++r) {
            const float v = scratch[r * 33 + lane];
            mx = fmaxf(mx, v);
            s += v;
          }
          const float mean = s / (float)nv;
          float se = 0.f, m2 = 0.f;
          for (int r = 0; r < nv; ++r) {
            const float v = scratch[r * 33 + lane];
            se += mx == -INFINITY ? 0.f : expf(v - mx);
            const float d = v - mean;
            m2 = fmaf(d, d, m2);
          }
          E.part[(row0 >> 5) * E.Np + n] = make_float4(mx, se, mean, m2);
        }
        __syncwarp();
      }
    } else if (PUSH) {
      // The tile's 128 rows belong to one owner rank (own % 128 == 0).  Each warp transposes its 32 x 32 blocks through
      // the shared-memory scratch so that every store instruction writes one 128-byte row segment into the owner's
      // window: plain NVLink stores, issued while the MMA warp is already accumulating the next tile.  The operand
      // scales are undone here (the ranks' scales differ); the owner adds the per-source slots in rank order.
      const int row0 = m0 + q * 32;
      const int owner = row0 / E.push_own;
      B2M_ASSERT(owner >= 0 && owner < kMaxPeers && E.push_dst[owner] != nullptr && (row0 + 31) / E.push_own == owner);
      float *dst = E.push_dst[owner] + ((int64_t)E.push_rank * E.push_own + (row0 - owner * E.push_own)) * E.Dp + nb;
      const float ru = E.r_unscale ? E.r_unscale[m] : 1.0f;   // lane r: scale of row r of this warp's 32 rows
      float *scratch = scratch_base + (warp - 2) * (32 * 33);
#pragma unroll
      for (int b = 0; b < CW / 32; ++b) {
#pragma unroll
        for (int j = 0; j < 32; ++j) scratch[lane * 33 + j] = acc[b * 32 + j] * ru;
        __syncwarp();
        const float ics = E.inv_col_scale ? E.inv_col_scale[nb + b * 32 + lane] : 1.0f;
#pragma unroll 8
        for (int r = 0; r < 32; ++r) dst[(int64_t)r * E.Dp + b * 32 + lane] = scratch[r * 33 + lane] * ics;
        __syncwarp();
      }
    } else {
      float *g = E.Gpart + ((int64_t)zs * E.Cp + m) * E.Dp + nb;
#pragma unroll
      for (int j = 0; j < CW; j += 4) *reinterpret_cast<float4 *>(g + j) = make_float4(acc[j], acc[j + 1], acc[j + 2], acc[j + 3]);
    }
    }
    // the writers themselves order their NVLink stores before anything that follows the kernel (the "partials stored"
    // flag is raised by the next kernel on this stream): a system-scope fence per pushing thread, once per launch
    if (PUSH) __threadfence_system();
  }
#undef B2M_DECODE_TILE

  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  if (NCTA == 2) cluster_sync_all(); else __syncthreads();   // no CTA of a pair may leave while its peer still signals it
  if (warp == 1) {
    if (NCTA == 2)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(C::TMEM_COLS));
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(C::TMEM_COLS));
  }
}

// ---------------------------------------------------------------- tensor maps
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void *p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// [rows, cols] row-major fp32, box = 32 columns (128 bytes) x box_rows rows, 128-byte swizzle.
// Encoded maps are cached by (base, rows, cols, box): a NUTS leaf would otherwise pay eight driver calls per
// value+gradient, which is visible at the small configurations where a leaf is ~100 us of device time.
int make_map_uncached(CUtensorMap *map, const void *base, int64_t rows, int64_t cols, int box_rows, bool f16);

struct MapKey {
  const void *base;
  int64_t rows, cols;
  int box;
  bool operator==(const MapKey &o) const { return base == o.base && rows == o.rows && cols == o.cols && box == o.box; }
};
struct MapSlot {
  MapKey key;
  CUtensorMap map;
};
static thread_local std::vector<MapSlot> tl_maps;

// `cols` in elements of the operand encoding (float for tf32, __half for f16: box is negative-coded as -box_rows)
int make_map(CUtensorMap *map, const void *base, int64_t rows, int64_t cols, int box_rows, bool f16 = false) {
  const MapKey key{base, rows, cols, f16 ? -box_rows : box_rows};
  for (const MapSlot &s : tl_maps)
    if (s.key == key) {
      *map = s.map;
      return 0;
    }
  if (int rc = make_map_uncached(map, base, rows, cols, box_rows, f16)) return rc;
  if (tl_maps.size() >= 256) tl_maps.clear();   // workspaces were reallocated many times: start over
  tl_maps.push_back(MapSlot{key, *map});
  return 0;
}

int make_map_uncached(CUtensorMap *map, const void *base, int64_t rows, int64_t cols, int box_rows, bool f16) {
  EncodeTiledFn fn = encode_fn();
  B2M_REQUIRE(fn != nullptr, "cuTensorMapEncodeTiled is not available from this driver");
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)cols * (f16 ? 2 : 4)};
  cuuint32_t box[2] = {(cuuint32_t)(f16 ? 64 : 32), (cuuint32_t)box_rows};   // one 128-byte swizzle row of K
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void *>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r));
    return 2;
  }
  return 0;
}

// ---------------------------------------------------------------- per-launch timing (bench.py's roofline)
struct Prof {
  bool on = false;
  // [0] = K5 (residual epilogue), [1] = K6 (gradient), [2] = NUTS state kernel, [3] = peer wait kernel, [4] = peer signal
  // kernel: start, stop, start, ...
  std::vector<cudaEvent_t> ev[5];
} g_prof;

template <int BLOCK_N, int MODE, int NCTA, bool F16>
int launch_tc_n(const CUtensorMap &Ah, const CUtensorMap &Al, const CUtensorMap &Bh, const CUtensorMap &Bl, dim3 grid,
                int kb_total, int kb_per_split, const EpiParams &E, cudaStream_t st, int chunk_kb, int mma_mask,
                int prof_kind) {
  using C = Cfg<BLOCK_N, NCTA>;
  constexpr bool RESID = MODE == 1 || MODE == 3 || MODE == 4 || MODE == 5;
  auto kernel = tc_gemm_kernel<BLOCK_N, MODE, NCTA, F16>;
  constexpr int SMEM = C::SMEM_BYTES + (MODE != 0 ? NUM_EPI_WARPS * 32 * 33 * 4 : 0);
  // per device: the attribute belongs to the function on the current device.  Setting it again is harmless, so a plain
  // atomic flag is enough for concurrent first calls from several threads.
  static std::atomic<bool> configured[64];
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || !configured[dev].load(std::memory_order_acquire)) {
    B2M_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    if (dev >= 0 && dev < 64) configured[dev].store(true, std::memory_order_release);
  }
  // `grid` arrives as (128-row tiles, column tiles, K splits); the launch is one persistent CTA group per SM (pair)
  const int Tm = (int)grid.x / NCTA, Tn = (int)grid.y, n_tiles = Tm * Tn * (int)grid.z;
  const int n_groups = n_tiles < 148 / NCTA ? n_tiles : 148 / NCTA;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (g_prof.on) {
    B2M_CHECK_CUDA(cudaEventCreate(&e0));
    B2M_CHECK_CUDA(cudaEventCreate(&e1));
    B2M_CHECK_CUDA(cudaEventRecord(e0, st));
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(n_groups * NCTA), 1, 1);
  cfg.blockDim = dim3(NUM_THREADS);
  cfg.dynamicSmemBytes = SMEM;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = NCTA;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = NCTA == 2 ? 1 : 0;
  B2M_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kernel, Ah, Al, Bh, Bl, kb_total, kb_per_split, chunk_kb, mma_mask, Tm, Tn, n_tiles, E));
  if (g_prof.on) {
    B2M_CHECK_CUDA(cudaEventRecord(e1, st));
    const int k = prof_kind >= 0 ? prof_kind : (RESID ? 0 : 1);
    g_prof.ev[k].push_back(e0);
    g_prof.ev[k].push_back(e1);
  }
  ++g_launches;
  B2M_CHECK_CUDA(cudaGetLastError());
  return 0;
}

template <int BLOCK_N, int MODE>
int launch_tc(int ncta, const CUtensorMap &Ah, const CUtensorMap &Al, const CUtensorMap &Bh, const CUtensorMap &Bl,
              dim3 grid, int kb_total, int kb_per_split, const EpiParams &E, cudaStream_t st,
              int chunk_kb = DEFAULT_CHUNK_KB, int mma_mask = 7, bool f16 = false, int prof_kind = -1) {
  if constexpr (MODE == 2) {   // the push epilogue exists for the shape it is used with: fp16 encoding, CTA pairs
    B2M_REQUIRE(f16 && ncta == 2, "K6 push epilogue: needs the fp16 encoding and whole 256-row tiles");
    return launch_tc_n<BLOCK_N, 2, 2, true>(Ah, Al, Bh, Bl, grid, kb_total, kb_per_split, E, st, chunk_kb, mma_mask, prof_kind);
  } else {
    if (f16) {
      if (ncta == 2) return launch_tc_n<BLOCK_N, MODE, 2, true>(Ah, Al, Bh, Bl, grid, kb_total, kb_per_split, E, st, chunk_kb, mma_mask, prof_kind);
      return launch_tc_n<BLOCK_N, MODE, 1, true>(Ah, Al, Bh, Bl, grid, kb_total, kb_per_split, E, st, chunk_kb, mma_mask, prof_kind);
    }
    if (ncta == 2) return launch_tc_n<BLOCK_N, MODE, 2, false>(Ah, Al, Bh, Bl, grid, kb_total, kb_per_split, E, st, chunk_kb, mma_mask, prof_kind);
    return launch_tc_n<BLOCK_N, MODE, 1, false>(Ah, Al, Bh, Bl, grid, kb_total, kb_per_split, E, st, chunk_kb, mma_mask, prof_kind);
  }
}

}  // namespace

bool tc_available() { return encode_fn() != nullptr; }

void tc_profile(bool enable) {
  for (auto &v : g_prof.ev) {
    for (cudaEvent_t e : v) cudaEventDestroy(e);
    v.clear();
  }
  g_prof.on = enable;
}

// bracket one launch of kind 2..4 (the per-chain kernels of the fused NUTS loop) with events while profiling is on
void prof_mark(int kind, cudaStream_t st) {
  if (!g_prof.on || kind < 0 || kind >= 5) return;
  cudaEvent_t e = nullptr;
  if (cudaEventCreate(&e) != cudaSuccess) return;
  cudaEventRecord(e, st);
  g_prof.ev[kind].push_back(e);
}

// out = {total ms, launches} per kind, n_kinds of them, since tc_profile(true); synchronises the device
int tc_profile_read_n(double *out, int n_kinds) {
  B2M_CHECK_CUDA(cudaDeviceSynchronize());
  for (int k = 0; k < n_kinds && k < 5; ++k) {
    double ms = 0.0;
    for (size_t i = 0; i + 1 < g_prof.ev[k].size(); i += 2) {
      float t = 0.f;
      B2M_CHECK_CUDA(cudaEventElapsedTime(&t, g_prof.ev[k][i], g_prof.ev[k][i + 1]));
      ms += t;
    }
    out[2 * k] = ms;
    out[2 * k + 1] = (double)(g_prof.ev[k].size() / 2);
  }
  return 0;
}

// out4 = {K5 total ms, K5 launches, K6 total ms, K6 launches} since tc_profile(true); synchronises the device
int tc_profile_read(double *out4) {
  B2M_CHECK_CUDA(cudaDeviceSynchronize());
  for (int k = 0; k < 2; ++k) {
    double ms = 0.0;
    for (size_t i = 0; i + 1 < g_prof.ev[k].size(); i += 2) {
      float t = 0.f;
      B2M_CHECK_CUDA(cudaEventElapsedTime(&t, g_prof.ev[k][i], g_prof.ev[k][i + 1]));
      ms += t;
    }
    out4[2 * k] = ms;
    out4[2 * k + 1] = (double)(g_prof.ev[k].size() / 2);
  }
  return 0;
}

int grad_block_n(const GlmModel &g) { return g.Dp % 256 == 0 ? 256 : (g.Dp % 128 == 0 ? 128 : 64); }

// CTA pairs need whole 256-row tiles of chains
static int pair_mode(int64_t Cp) { return (Cp % 256 == 0) ? 2 : 1; }

// split-K factor of the gradient contraction over `kb` k-blocks (K6: K = Np; Gram form: K = Dp): enough CTAs to fill
// the 148 SMs in whole waves, each split at least 8 k-blocks deep
int grad_splits(const GlmModel &g, int64_t Cp, int kb) {
  const int64_t tiles = (Cp / BLOCK_M) * (g.Dp / grad_block_n(g));   // CTAs per split
  int max_s = kb / 8 > 0 ? kb / 8 : 1;
  if (max_s > 32) max_s = 32;
  int best = 1;
  double best_eff = 0.0;
  for (int s = 1; s <= max_s; ++s) {
    const int64_t ctas = tiles * s;
    const int64_t waves = (ctas + 147) / 148;
    // efficiency of the last wave, minus a small charge per split for writing / re-reading the partials
    const double eff = (double)ctas / (double)(waves * 148) - 0.004 * (s - 1);
    if (eff > best_eff + 1e-9) { best_eff = eff; best = s; }
  }
  return best;
}

int contraction_splits(const GlmModel &g, int64_t Cp) {
  return grad_splits(g, Cp, (g.form == kFormGram ? g.Dp : g.Np) / (g.use_tc == 2 ? 64 : 32));
}

int tc_gemm_resid(GlmModel &g, int64_t Cp, cudaStream_t st) {
  const int ncta = pair_mode(Cp);
  const bool f16 = g.use_tc == 2;
  const int bk = f16 ? 64 : 32;
  const void *A_h = f16 ? (const void *)g.B16h : (const void *)g.Bh, *A_l = f16 ? (const void *)g.B16l : (const void *)g.Bl;
  const void *B_h = f16 ? (const void *)g.X16h : (const void *)g.Xh, *B_l = f16 ? (const void *)g.X16l : (const void *)g.Xl;
  CUtensorMap Ah, Al, Bh, Bl;
  if (make_map(&Ah, A_h, Cp, g.Dp, BLOCK_M, f16) || make_map(&Al, A_l, Cp, g.Dp, BLOCK_M, f16) ||
      make_map(&Bh, B_h, g.Np, g.Dp, 256 / ncta, f16) || make_map(&Bl, B_l, g.Np, g.Dp, 256 / ncta, f16))
    return 2;
  EpiParams E{};
  E.y = g.y0; E.inv_var = g.inv_var; E.ss_part = g.ss_part; E.Cp = Cp; E.Np = g.Np;
  E.skip_flag = g.skip_flag; E.skip_target = g.skip_target;
  E.Rh = f16 ? (void *)g.R16h : (void *)g.Rh;
  E.Rl = f16 ? (void *)g.R16l : (void *)g.Rl;
  E.a_unscale = g.a_unscale; E.r_scale = g.r_scale;
  E.N_valid = g.N; E.loc_const = 0.f; E.weight = g.weight;   // y0 is already centred and shifted (glm.cu)
  const bool logit = g.lik == kLikLogit;
  if (logit) { E.y = g.y; E.eta0 = g.y0; }   // labels, and the centring c + X beta0
  dim3 grid((unsigned)(Cp / BLOCK_M), g.Np / 256, 1);
  // promotion interval: 128 values of K for tf32; 256 for fp16 -- the MMAs of a tile take half as long there, and the
  // longer chunk lets the issuer run far enough into the next tile to cover the epilogue (measured at C4: 4.28 ->
  // 4.12 ms per evaluation, gradient error 1.3e-6 -> 2.1e-6; K5's accumulators only hold X (beta - beta0))
  // fp16 encoding with K >= 512: two chunks of 8 k-blocks (512 values of K) per tile instead of four of 4 -- TMEM holds two
  // chunk accumulators, so the issuer can then run a WHOLE tile ahead of the residual epilogue instead of half a tile
  // (measured at C4: K5 1.94 -> 1.89 ms; gradient error vs float64 unchanged at 2e-6, full-size test green)
  const int ck = (f16 && g.Dp / bk >= 8) ? 8 : DEFAULT_CHUNK_KB;
  if (logit) return launch_tc<256, 3>(ncta, Ah, Al, Bh, Bl, grid, g.Dp / bk, g.Dp / bk, E, st, ck, 7, f16);
  return launch_tc<256, 1>(ncta, Ah, Al, Bh, Bl, grid, g.Dp / bk, g.Dp / bk, E, st, ck, 7, f16);
}

// K5 over a batch of posterior draws with the statistics epilogue: the operand set-up and tile schedule of
// tc_gemm_resid, no residual operand, per-observation partials of 32 draws into `part` [Cp / 32, Np].  Timed in the
// K5 slot of the profile.
int tc_gemm_stats(GlmModel &g, int64_t Cp, int64_t rows_valid, float4 *part, cudaStream_t st) {
  const int ncta = pair_mode(Cp);
  const bool f16 = g.use_tc == 2;
  const int bk = f16 ? 64 : 32;
  const void *A_h = f16 ? (const void *)g.B16h : (const void *)g.Bh, *A_l = f16 ? (const void *)g.B16l : (const void *)g.Bl;
  const void *B_h = f16 ? (const void *)g.X16h : (const void *)g.Xh, *B_l = f16 ? (const void *)g.X16l : (const void *)g.Xl;
  CUtensorMap Ah, Al, Bh, Bl;
  if (make_map(&Ah, A_h, Cp, g.Dp, BLOCK_M, f16) || make_map(&Al, A_l, Cp, g.Dp, BLOCK_M, f16) ||
      make_map(&Bh, B_h, g.Np, g.Dp, 256 / ncta, f16) || make_map(&Bl, B_l, g.Np, g.Dp, 256 / ncta, f16))
    return 2;
  EpiParams E{};
  E.y = g.y0; E.inv_var = g.inv_var; E.Cp = Cp; E.Np = g.Np;
  E.a_unscale = g.a_unscale;
  E.N_valid = g.N; E.weight = g.weight;
  E.part = part; E.rows_valid = rows_valid;
  const bool logit = g.lik == kLikLogit;
  if (logit) { E.y = g.y; E.eta0 = g.y0; }
  dim3 grid((unsigned)(Cp / BLOCK_M), g.Np / 256, 1);
  const int ck = (f16 && g.Dp / bk >= 8) ? 8 : DEFAULT_CHUNK_KB;   // as tc_gemm_resid
  if (logit) return launch_tc<256, 5>(ncta, Ah, Al, Bh, Bl, grid, g.Dp / bk, g.Dp / bk, E, st, ck, 7, f16);
  return launch_tc<256, 4>(ncta, Ah, Al, Bh, Bl, grid, g.Dp / bk, g.Dp / bk, E, st, ck, 7, f16);
}

int tc_gemm_grad(GlmModel &g, int64_t Cp, cudaStream_t st) {
  const int ncta = pair_mode(Cp);
  const bool f16 = g.use_tc == 2;
  const int bk = f16 ? 64 : 32;
  const int bn = grad_block_n(g);
  const int kb_total = g.Np / bk;
  const int splits = grad_splits(g, Cp, kb_total);
  const int kb_per = (kb_total + splits - 1) / splits;
  const void *A_h = f16 ? (const void *)g.R16h : (const void *)g.Rh, *A_l = f16 ? (const void *)g.R16l : (const void *)g.Rl;
  const void *B_h = f16 ? (const void *)g.XT16h : (const void *)g.XTh, *B_l = f16 ? (const void *)g.XT16l : (const void *)g.XTl;
  CUtensorMap Ah, Al, Bh, Bl;
  if (make_map(&Ah, A_h, Cp, g.Np, BLOCK_M, f16) || make_map(&Al, A_l, Cp, g.Np, BLOCK_M, f16) ||
      make_map(&Bh, B_h, g.Dp, g.Np, bn / ncta, f16) || make_map(&Bl, B_l, g.Dp, g.Np, bn / ncta, f16))
    return 2;
  EpiParams E{};
  E.Gpart = g.G; E.Cp = Cp; E.Dp = g.Dp;
  E.skip_flag = g.skip_flag; E.skip_target = g.skip_target;
  dim3 grid((unsigned)(Cp / BLOCK_M), g.Dp / bn, (unsigned)((kb_total + kb_per - 1) / kb_per));
  g.g_splits = (int)grid.z;
  const int ck = f16 ? DEFAULT_CHUNK_KB / 2 : DEFAULT_CHUNK_KB;
  if (bn == 256) return launch_tc<256, 0>(ncta, Ah, Al, Bh, Bl, grid, kb_total, kb_per, E, st, ck, 7, f16);
  if (bn == 128) return launch_tc<128, 0>(ncta, Ah, Al, Bh, Bl, grid, kb_total, kb_per, E, st, ck, 7, f16);
  return launch_tc<64, 0>(ncta, Ah, Al, Bh, Bl, grid, kb_total, kb_per, E, st, ck, 7, f16);
}

// Gram form: P = (packed delta rows) G~, [Cp, Dp] x [Dp, Dp] -- the K6 kernel body with the packed rows of K5 as the A
// operand and the Gram halves as the B operand (K = Dp).  Its launch is the only contraction of an evaluation and is timed
// in the K5 slot of the profile (b2m_profile_read): readers that sum K5 + K6 get the contraction time of one evaluation
// and, with no K6 entries, count one launch per evaluation.
int tc_gemm_gram(GlmModel &g, int64_t Cp, cudaStream_t st) {
  B2M_REQUIRE(g.form == kFormGram && g.Gmh && g.Gml, "tc_gemm_gram: the model has no Gram operand");
  const int ncta = pair_mode(Cp);
  const bool f16 = g.use_tc == 2;
  const int bk = f16 ? 64 : 32;
  const int bn = grad_block_n(g);
  const int kb_total = g.Dp / bk;
  const int splits = grad_splits(g, Cp, kb_total);
  const int kb_per = (kb_total + splits - 1) / splits;
  const void *A_h = f16 ? (const void *)g.B16h : (const void *)g.Bh, *A_l = f16 ? (const void *)g.B16l : (const void *)g.Bl;
  CUtensorMap Ah, Al, Bh, Bl;
  if (make_map(&Ah, A_h, Cp, g.Dp, BLOCK_M, f16) || make_map(&Al, A_l, Cp, g.Dp, BLOCK_M, f16) ||
      make_map(&Bh, g.Gmh, g.Dp, g.Dp, bn / ncta, f16) || make_map(&Bl, g.Gml, g.Dp, g.Dp, bn / ncta, f16))
    return 2;
  EpiParams E{};
  E.Gpart = g.G; E.Cp = Cp; E.Dp = g.Dp;
  E.skip_flag = g.skip_flag; E.skip_target = g.skip_target;
  dim3 grid((unsigned)(Cp / BLOCK_M), g.Dp / bn, (unsigned)((kb_total + kb_per - 1) / kb_per));
  g.g_splits = (int)grid.z;
  const int ck = f16 ? DEFAULT_CHUNK_KB / 2 : DEFAULT_CHUNK_KB;
  if (bn == 256) return launch_tc<256, 0>(ncta, Ah, Al, Bh, Bl, grid, kb_total, kb_per, E, st, ck, 7, f16, 0);
  if (bn == 128) return launch_tc<128, 0>(ncta, Ah, Al, Bh, Bl, grid, kb_total, kb_per, E, st, ck, 7, f16, 0);
  return launch_tc<64, 0>(ncta, Ah, Al, Bh, Bl, grid, kb_total, kb_per, E, st, ck, 7, f16, 0);
}

// K6 of a peer-sliced observation shard: one K pass over the rank's rows (no split-K: every output tile is produced
// once and leaves through the epilogue), tiles pushed into the owners' windows.
int tc_gemm_grad_push(GlmModel &g, int64_t Cp, cudaStream_t st) {
  const PeerWindow &w = g.pw;
  B2M_REQUIRE(w.nranks >= 2 && g.use_tc == 2 && Cp == w.C && Cp % 256 == 0 && w.own % 128 == 0,
              "K6 push epilogue: needs an attached peer window, the fp16 encoding and a full batch");
  const int bk = 64, bn = grad_block_n(g);
  const int kb_total = g.Np / bk;
  CUtensorMap Ah, Al, Bh, Bl;
  if (make_map(&Ah, g.R16h, Cp, g.Np, BLOCK_M, true) || make_map(&Al, g.R16l, Cp, g.Np, BLOCK_M, true) ||
      make_map(&Bh, g.XT16h, g.Dp, g.Np, bn / 2, true) || make_map(&Bl, g.XT16l, g.Dp, g.Np, bn / 2, true))
    return 2;
  EpiParams E{};
  E.Cp = Cp; E.Dp = g.Dp;
  E.push_own = (int)w.own; E.push_rank = w.rank;
  for (int s = 0; s < w.nranks; ++s) E.push_dst[s] = reinterpret_cast<float *>(w.base[s] + w.off_g);
  E.r_unscale = g.r_unscale; E.inv_col_scale = g.inv_col_scale;
  dim3 grid((unsigned)(Cp / BLOCK_M), g.Dp / bn, 1);
  g.g_splits = 1;
  const int ck = DEFAULT_CHUNK_KB / 2;
  if (bn == 256) return launch_tc<256, 2>(2, Ah, Al, Bh, Bl, grid, kb_total, kb_total, E, st, ck, 7, true);
  if (bn == 128) return launch_tc<128, 2>(2, Ah, Al, Bh, Bl, grid, kb_total, kb_total, E, st, ck, 7, true);
  return launch_tc<64, 2>(2, Ah, Al, Bh, Bl, grid, kb_total, kb_total, E, st, ck, 7, true);
}


// ---------------------------------------------------------------- raw 3xTF32 GEMM for experiments / tests
__global__ void split_kernel(const float *__restrict__ x, int64_t n, float *hi, float *lo) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) split_tf32(x[i], hi[i], lo[i]);
}

int debug_tc_gemm(const float *A, const float *Bm, int M, int N, int K, float *Cout, int chunk_kb, int mma_mask,
                  cudaStream_t st) {
  B2M_REQUIRE(M % BLOCK_M == 0 && N % 64 == 0 && K % BLOCK_K == 0, "debug_tc_gemm: M%128, N%64, K%32 must be 0");
  float *Ah, *Al, *Bh, *Bl;
  B2M_CHECK_CUDA(cudaMalloc(&Ah, sizeof(float) * M * (size_t)K));
  B2M_CHECK_CUDA(cudaMalloc(&Al, sizeof(float) * M * (size_t)K));
  B2M_CHECK_CUDA(cudaMalloc(&Bh, sizeof(float) * N * (size_t)K));
  B2M_CHECK_CUDA(cudaMalloc(&Bl, sizeof(float) * N * (size_t)K));
  split_kernel<<<(unsigned)(((size_t)M * K + 255) / 256), 256, 0, st>>>(A, (int64_t)M * K, Ah, Al);
  split_kernel<<<(unsigned)(((size_t)N * K + 255) / 256), 256, 0, st>>>(Bm, (int64_t)N * K, Bh, Bl);
  const int bn = N % 256 == 0 ? 256 : (N % 128 == 0 ? 128 : 64);
  const int ncta = pair_mode(M);
  CUtensorMap mAh, mAl, mBh, mBl;
  int rc = make_map(&mAh, Ah, M, K, BLOCK_M) || make_map(&mAl, Al, M, K, BLOCK_M) || make_map(&mBh, Bh, N, K, bn / ncta) ||
           make_map(&mBl, Bl, N, K, bn / ncta);
  if (!rc) {
    EpiParams E{};
    E.Gpart = Cout; E.Cp = M; E.Dp = N;
    dim3 grid(M / BLOCK_M, N / bn, 1);
    if (bn == 256) rc = launch_tc<256, 0>(ncta, mAh, mAl, mBh, mBl, grid, K / BLOCK_K, K / BLOCK_K, E, st, chunk_kb, mma_mask);
    else if (bn == 128) rc = launch_tc<128, 0>(ncta, mAh, mAl, mBh, mBl, grid, K / BLOCK_K, K / BLOCK_K, E, st, chunk_kb, mma_mask);
    else rc = launch_tc<64, 0>(ncta, mAh, mAl, mBh, mBl, grid, K / BLOCK_K, K / BLOCK_K, E, st, chunk_kb, mma_mask);
  }
  cudaStreamSynchronize(st);
  cudaFree(Ah); cudaFree(Al); cudaFree(Bh); cudaFree(Bl);
  return rc ? 2 : 0;
}

}  // namespace b2m

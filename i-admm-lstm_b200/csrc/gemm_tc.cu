// Plain "NT" GEMM on the tensor cores for the training backward pass:
//     C[M,N] = scale * A[M,K] * B[N,K]^T          (fp32 result, fp32-class accuracy)
// Both operands arrive as fp16 hi/lo images of power-of-two scaled fp32 data, K-major ([rows][K]); the three
// products A_lo B_hi + A_hi B_lo + A_hi B_hi accumulate in fp32 in tensor memory (same split as the forward gate
// kernel's IADMM_GATES_TC_3XFP16 mode) and `scale` undoes the operand scalings.
// Used for the two gate-product adjoints of one iteration (models/lstm.py:74-77 under autograd):
//     H_bar = D U^T        A = D  [rows,4h],   B = U   [h,4h]    (K = 4h)
//     U_bar = H^T D        A = H^T [h,rows],   B = D^T [4h,rows] (K = rows)
// plus the conversion kernels that produce those images (row-wise split, and split + transpose).
// Same warp-specialised structure as gates_tc_kernel: TMA producer warp, single-thread tcgen05.mma issuer,
// 8 epilogue warps draining a double-buffered TMEM accumulator; tile 128 x 256, 64-wide K stages.
#include "common.cuh"
#include "tc_ptx.cuh"

namespace iadmm {

constexpr int kGmBN = 256;
constexpr int kGmBK = 64;
constexpr int kGmEpiWarps = 8;
constexpr int kGmThreads = 32 * (2 + kGmEpiWarps);
constexpr int kGmABytes = kTcBM * kGmBK * 2;     // 16 KB
constexpr int kGmBBytes = kGmBN * kGmBK * 2;     // 32 KB
constexpr int kGmStageBytes = 2 * (kGmABytes + kGmBBytes);   // 96 KB
constexpr int kGmStages = 2;

struct GemmParams {
  float* C;                // splits == 1: the result; splits > 1: partial results [splits][M][ldc]
  const float* scale;      // device scalar
  long M, N, K, ldc;
  int n_tiles, k_blocks;
  int splits, kb_per_split;   // split-K: work unit = (tile, split), split s covers K blocks [s*kb_per_split, ...)
  long num_tiles;             // output tiles; work units = num_tiles * splits
  int prod_mask;              // which of the products are issued: 1 = A_lo B_hi, 2 = A_hi B_lo, 4 = A_hi B_hi (7 = all)
};

__global__ void __launch_bounds__(kGmThreads, 1)
tc_gemm_nt_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                  const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo,
                  const GemmParams P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)kGmStages * kGmStageBytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + kGmStages;
  uint64_t* tfull_bar = bars + 2 * kGmStages;
  uint64_t* tempty_bar = bars + 2 * kGmStages + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kGmStages + 4);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a_hi); tma_prefetch_desc(&map_a_lo); tma_prefetch_desc(&map_b_hi); tma_prefetch_desc(&map_b_lo);
    for (int s = 0; s < kGmStages; ++s) { mbar_init(smem_u32(&full_bar[s]), 1); mbar_init(smem_u32(&empty_bar[s]), 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(smem_u32(&tfull_bar[b]), 1); mbar_init(smem_u32(&tempty_bar[b]), kGmEpiWarps); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (long unit = blockIdx.x; unit < P.num_tiles * P.splits; unit += gridDim.x) {
        const long tile = unit / P.splits;
        const int sp = (int)(unit - tile * P.splits);
        const int nt = (int)(tile % P.n_tiles);
        const long mt = tile / P.n_tiles;
        const int row0 = (int)(mt * kTcBM), col0 = nt * kGmBN;
        const int kb_end = min(P.k_blocks, (sp + 1) * P.kb_per_split);
        for (int kb = sp * P.kb_per_split; kb < kb_end; ++kb) {
          mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1);
          const uint32_t fb = smem_u32(&full_bar[stage]);
          mbar_expect_tx(fb, kGmStageBytes);
          const uint32_t sb = smem_u32(smem + (size_t)stage * kGmStageBytes);
          const int k0 = kb * kGmBK;
          tma_load_2d(sb, &map_a_hi, fb, k0, row0);
          tma_load_2d(sb + kGmABytes, &map_a_lo, fb, k0, row0);
          tma_load_2d(sb + 2 * kGmABytes, &map_b_hi, fb, k0, col0);
          tma_load_2d(sb + 2 * kGmABytes + kGmBBytes, &map_b_lo, fb, k0, col0);
          if (++stage == kGmStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      long it = 0;
      for (long unit = blockIdx.x; unit < P.num_tiles * P.splits; unit += gridDim.x, ++it) {
        const long tile = unit / P.splits;
        const int sp = (int)(unit - tile * P.splits);
        const int kb_end = min(P.k_blocks, (sp + 1) * P.kb_per_split);
        const int nt = (int)(tile % P.n_tiles);
        const int n_cols = (int)min((long)kGmBN, P.N - (long)nt * kGmBN);
        const uint32_t idesc = make_idesc_f16(n_cols);
        const int buf = (int)(it & 1);
        const uint32_t use = (uint32_t)(it >> 1);
        mbar_wait(smem_u32(&tempty_bar[buf]), (use & 1) ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(buf * kGmBN);
        uint32_t acc = 0;
        for (int kb = sp * P.kb_per_split; kb < kb_end; ++kb) {
          mbar_wait(smem_u32(&full_bar[stage]), phase);
          tc_fence_after();
          const uint32_t sb = smem_u32(smem + (size_t)stage * kGmStageBytes);
          const long k_len = min((long)kGmBK, P.K - (long)kb * kGmBK);
          const int k_steps = (int)((k_len + kTcUK - 1) / kTcUK);
          for (int ks = 0; ks < k_steps; ++ks) {
            const uint32_t koff = (uint32_t)(ks * kTcUK * 2);
            const uint64_t a_hi = make_smem_desc_sw128(sb + koff);
            const uint64_t a_lo = make_smem_desc_sw128(sb + kGmABytes + koff);
            const uint64_t b_hi = make_smem_desc_sw128(sb + 2 * kGmABytes + koff);
            const uint64_t b_lo = make_smem_desc_sw128(sb + 2 * kGmABytes + kGmBBytes + koff);
            tc_mma_f16(d_tmem, a_lo, b_hi, idesc, acc); acc = 1;
            tc_mma_f16(d_tmem, a_hi, b_lo, idesc, 1);
            tc_mma_f16(d_tmem, a_hi, b_hi, idesc, 1);
          }
          tc_commit(smem_u32(&empty_bar[stage]));
          if (++stage == kGmStages) { stage = 0; phase ^= 1; }
        }
        tc_commit(smem_u32(&tfull_bar[buf]));
      }
    }
  } else {
    const int ew = warp - 2;
    const int quarter = warp & 3;
    const int half = (ew >= 4) ? 1 : 0;
    const float scale = *P.scale;
    long it = 0;
    for (long unit = blockIdx.x; unit < P.num_tiles * P.splits; unit += gridDim.x, ++it) {
      const long tile = unit / P.splits;
      const int sp = (int)(unit - tile * P.splits);
      const int nt = (int)(tile % P.n_tiles);
      const long mt = tile / P.n_tiles;
      const int buf = (int)(it & 1);
      const uint32_t use = (uint32_t)(it >> 1);
      const long row = mt * kTcBM + quarter * 32 + lane;
      mbar_wait(smem_u32(&tfull_bar[buf]), use & 1);
      tc_fence_after();
#pragma unroll 1
      for (int cc = 0; cc < 4; ++cc) {
        const int chunk = half * 4 + cc;
        const long col0 = (long)nt * kGmBN + chunk * 32;
        uint32_t v[32];
        tc_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(buf * kGmBN + chunk * 32), v);
        tc_wait_ld();
        if (row < P.M) {
          float* crow = P.C + ((size_t)sp * P.M + row) * P.ldc + col0;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            if (col0 + q * 8 < P.N) {            // N % 8 == 0
              float4 o0 = make_float4(__uint_as_float(v[q * 8 + 0]) * scale, __uint_as_float(v[q * 8 + 1]) * scale,
                                      __uint_as_float(v[q * 8 + 2]) * scale, __uint_as_float(v[q * 8 + 3]) * scale);
              float4 o1 = make_float4(__uint_as_float(v[q * 8 + 4]) * scale, __uint_as_float(v[q * 8 + 5]) * scale,
                                      __uint_as_float(v[q * 8 + 6]) * scale, __uint_as_float(v[q * 8 + 7]) * scale);
              *reinterpret_cast<float4*>(crow + q * 8) = o0;
              *reinterpret_cast<float4*>(crow + q * 8 + 4) = o1;
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&tempty_bar[buf]));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

// A_hi/A_lo: [M][lda], B_hi/B_lo: [N][ldb] fp16 K-major; lda, ldb multiples of 8; N multiple of 16; C fp32 [M][ldc], ldc % 4 == 0
// ================================================================================================
// CTA-pair variant (cta_group::2): tile = 256 rows x 256 columns over two SMs, the barrier protocol of
// gates_tc_pair_kernel (gates_tc.cu): each CTA loads its own 128 rows of A and HALF of the B tile, the leader issues
// M = 256 MMAs that read both halves; `full` lives in the leader and counts the TMA bytes of BOTH CTAs, `empty` and `tmem_full`
// are signalled in both CTAs by multicast tcgen05.commit, `tmem_empty` lives in the leader and collects the epilogue warps of
// both CTAs through the cluster window.  Per SM and K block 64 KB of operands feed 12 MMA-halves of 256x256x16 instead of 96 KB
// for 12 MMAs of 128x256x16: the single-CTA form is L2->SM fill bound with 4-byte (hi + lo) operands.
// ================================================================================================
constexpr int kGpABytes = kTcBM * kGmBK * 2;            // 16 KB: this CTA's 128 rows of A (one of hi / lo)
constexpr int kGpBBytes = (kGmBN / 2) * kGmBK * 2;      // 16 KB: this CTA's half of the B tile (one of hi / lo)
constexpr int kGpStageBytes = 2 * (kGpABytes + kGpBBytes);   // 64 KB
constexpr int kGpStages = 3;
constexpr int kGpBoxRows = 64;                          // B halves are fetched in 64-row TMA boxes

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGmThreads, 1)
tc_gemm_nt_pair_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                       const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo,
                       const GemmParams P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)kGpStages * kGpStageBytes);
  uint64_t* full_bar = bars;                         // [stages]  (leader's copy is the live one)
  uint64_t* empty_bar = bars + kGpStages;            // [stages]  both CTAs
  uint64_t* tfull_bar = bars + 2 * kGpStages;        // [2]       both CTAs
  uint64_t* tempty_bar = bars + 2 * kGpStages + 2;   // [2]       leader's copy is the live one
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kGpStages + 4);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a_hi); tma_prefetch_desc(&map_a_lo); tma_prefetch_desc(&map_b_hi); tma_prefetch_desc(&map_b_lo);
    for (int s = 0; s < kGpStages; ++s) { mbar_init(smem_u32(&full_bar[s]), 1); mbar_init(smem_u32(&empty_bar[s]), 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(smem_u32(&tfull_bar[b]), 1); mbar_init(smem_u32(&tempty_bar[b]), 2 * kGmEpiWarps); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::);
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const long pair = blockIdx.x / 2, num_pairs = gridDim.x / 2;
  const long units = P.num_tiles * P.splits;          // num_tiles counts 256-row tiles here

  if (warp == 0) {
    // ===================== TMA producer (every CTA) =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (long unit = pair; unit < units; unit += num_pairs) {
        const long tile = unit / P.splits;
        const int sp = (int)(unit - tile * P.splits);
        const int nt = (int)(tile % P.n_tiles);
        const long mt = tile / P.n_tiles;
        const int n_cols = (int)min((long)kGmBN, P.N - (long)nt * kGmBN);
        const int row0 = (int)(mt * (2 * kTcBM)) + (int)rank * kTcBM;          // this CTA's 128 rows of A
        const int col0 = nt * kGmBN + (int)rank * (n_cols / 2);                // first row of this CTA's half of the B tile
        const int b_boxes = (n_cols / 2 + kGpBoxRows - 1) / kGpBoxRows;
        const int kb_end = min(P.k_blocks, (sp + 1) * P.kb_per_split);
        for (int kb = sp * P.kb_per_split; kb < kb_end; ++kb) {
          mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1);
          const uint32_t fb_local = smem_u32(&full_bar[stage]);
          if (leader) mbar_expect_tx(fb_local, 2u * (2u * kGpABytes + (uint32_t)b_boxes * 2u * (kGpBoxRows * kGmBK * 2)));
          const uint32_t fb = map_to_cta(fb_local, 0);
          const uint32_t sb = smem_u32(smem + (size_t)stage * kGpStageBytes);
          const int k0 = kb * kGmBK;
          tma_load_2d_pair(sb, &map_a_hi, fb, k0, row0);
          tma_load_2d_pair(sb + kGpABytes, &map_a_lo, fb, k0, row0);
          for (int bx = 0; bx < b_boxes; ++bx) {
            tma_load_2d_pair(sb + 2 * kGpABytes + (uint32_t)bx * (kGpBoxRows * 128), &map_b_hi, fb, k0, col0 + bx * kGpBoxRows);
            tma_load_2d_pair(sb + 2 * kGpABytes + kGpBBytes + (uint32_t)bx * (kGpBoxRows * 128), &map_b_lo, fb, k0, col0 + bx * kGpBoxRows);
          }
          if (++stage == kGpStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (leader && lane == 0) {
      int stage = 0; uint32_t phase = 0;
      long it = 0;
      for (long unit = pair; unit < units; unit += num_pairs, ++it) {
        const long tile = unit / P.splits;
        const int sp = (int)(unit - tile * P.splits);
        const int nt = (int)(tile % P.n_tiles);
        const int n_cols = (int)min((long)kGmBN, P.N - (long)nt * kGmBN);
        const uint32_t idesc = make_idesc_f16(n_cols, 2 * kTcBM);
        const int buf = (int)(it & 1);
        const uint32_t use = (uint32_t)(it >> 1);
        const int kb_end = min(P.k_blocks, (sp + 1) * P.kb_per_split);
        mbar_wait(smem_u32(&tempty_bar[buf]), (use & 1) ^ 1);     // both CTAs' epilogues drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(buf * kGmBN);
        uint32_t acc = 0;
        for (int kb = sp * P.kb_per_split; kb < kb_end; ++kb) {
          mbar_wait(smem_u32(&full_bar[stage]), phase);
          tc_fence_after();
          const uint32_t sb = smem_u32(smem + (size_t)stage * kGpStageBytes);
          const long k_len = min((long)kGmBK, P.K - (long)kb * kGmBK);
          const int k_steps = (int)((k_len + kTcUK - 1) / kTcUK);
          for (int ks = 0; ks < k_steps; ++ks) {
            const uint32_t koff = (uint32_t)(ks * kTcUK * 2);
            const uint64_t a_hi = make_smem_desc_sw128(sb + koff);
            const uint64_t a_lo = make_smem_desc_sw128(sb + kGpABytes + koff);
            const uint64_t b_hi = make_smem_desc_sw128(sb + 2 * kGpABytes + koff);
            const uint64_t b_lo = make_smem_desc_sw128(sb + 2 * kGpABytes + kGpBBytes + koff);
            if (P.prod_mask & 1) { tc_mma_f16_pair(d_tmem, a_lo, b_hi, idesc, acc); acc = 1; }
            if (P.prod_mask & 2) { tc_mma_f16_pair(d_tmem, a_hi, b_lo, idesc, acc); acc = 1; }
            tc_mma_f16_pair(d_tmem, a_hi, b_hi, idesc, acc); acc = 1;
          }
          tc_commit_pair(smem_u32(&empty_bar[stage]), (uint16_t)3);   // frees the stage in both CTAs when the MMAs retire
          if (++stage == kGpStages) { stage = 0; phase ^= 1; }
        }
        tc_commit_pair(smem_u32(&tfull_bar[buf]), (uint16_t)3);       // accumulators complete in both CTAs
      }
    }
  } else {
    // ===================== epilogue (both CTAs, own 128 rows) =====================
    const int ew = warp - 2;
    const int quarter = warp & 3;
    const int half = (ew >= 4) ? 1 : 0;
    const float scale = *P.scale;
    long it = 0;
    for (long unit = pair; unit < units; unit += num_pairs, ++it) {
      const long tile = unit / P.splits;
      const int sp = (int)(unit - tile * P.splits);
      const int nt = (int)(tile % P.n_tiles);
      const long mt = tile / P.n_tiles;
      const int buf = (int)(it & 1);
      const uint32_t use = (uint32_t)(it >> 1);
      const long row = mt * (2 * kTcBM) + (long)rank * kTcBM + quarter * 32 + lane;
      mbar_wait(smem_u32(&tfull_bar[buf]), use & 1);
      tc_fence_after();
#pragma unroll 1
      for (int cc = 0; cc < 4; ++cc) {
        const int chunk = half * 4 + cc;
        const long col0 = (long)nt * kGmBN + chunk * 32;
        uint32_t v[32];
        tc_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(buf * kGmBN + chunk * 32), v);
        tc_wait_ld();
        if (row < P.M) {
          float* crow = P.C + ((size_t)sp * P.M + row) * P.ldc + col0;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            if (col0 + q * 8 < P.N) {            // N % 8 == 0
              float4 o0 = make_float4(__uint_as_float(v[q * 8 + 0]) * scale, __uint_as_float(v[q * 8 + 1]) * scale,
                                      __uint_as_float(v[q * 8 + 2]) * scale, __uint_as_float(v[q * 8 + 3]) * scale);
              float4 o1 = make_float4(__uint_as_float(v[q * 8 + 4]) * scale, __uint_as_float(v[q * 8 + 5]) * scale,
                                      __uint_as_float(v[q * 8 + 6]) * scale, __uint_as_float(v[q * 8 + 7]) * scale);
              *reinterpret_cast<float4*>(crow + q * 8) = o0;
              *reinterpret_cast<float4*>(crow + q * 8 + 4) = o1;
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(map_to_cta(smem_u32(&tempty_bar[buf]), 0));
    }
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

// sum of the split-K partials in a fixed order (deterministic): C[i] = ((p0 + p1) + p2) + ...
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const float4* __restrict__ part, float4* __restrict__ C, size_t count4, int splits) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count4) return;
  float4 a = part[i];
  for (int s = 1; s < splits; ++s) {
    const float4 b = part[(size_t)s * count4 + i];
    a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
  }
  C[i] = a;
}

// Split-K factor for a GEMM with few output tiles and a long K (U_bar = H^T D: 7 x 13 tiles, K = rows): the (tile, split)
// work units should fill whole waves of the persistent grid.  Picks the factor <= max_splits with the best wave efficiency
// (ties: the smaller one); every split keeps at least 8 K blocks.
int tc_gemm_pick_splits(long M, long N, long K, int num_sms, int max_splits) {
  // (the pair kernel works on 256-row tiles with one unit per pair of SMs: same wave arithmetic on num_sms / 2 pairs)
  const char* sw = dev_env("IADMM_GEMM_PAIR");
  const bool pair = num_sms >= 2 && !(sw && sw[0] == '0') && (N % 16 == 0);
  const long tile_rows = pair ? 2 * kTcBM : kTcBM;
  if (pair) num_sms /= 2;
  const long tiles = ((M + tile_rows - 1) / tile_rows) * ((N + kGmBN - 1) / kGmBN);
  const long k_blocks = (K + kGmBK - 1) / kGmBK;
  if (tiles >= 4L * num_sms) return 1;
  int best = 1;
  double best_eff = 0.0;
  for (int s = 1; s <= max_splits && k_blocks / s >= 8; ++s) {
    const long units = tiles * s;
    const long waves = (units + num_sms - 1) / num_sms;
    const double eff = (double)units / (double)(waves * num_sms);
    if (eff > best_eff + 1e-9) { best_eff = eff; best = s; }
  }
  return best;
}

// splits > 1: `part` must hold splits * M * ldc floats; C then receives the fixed-order sum of the partials
int launch_tc_gemm_nt(const __half* A_hi, const __half* A_lo, const __half* B_hi, const __half* B_lo, float* C,
                      const float* scale, long M, long N, long K, long lda, long ldb, long ldc, cudaStream_t st,
                      int splits, float* part, int prod_mask) {
  if (N % 16 != 0 || lda % 8 != 0 || ldb % 8 != 0 || ldc % 4 != 0) IADMM_FAIL(IADMM_ESHAPE, "tc_gemm: unsupported leading dimensions");
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) IADMM_FAIL(IADMM_ECUDA, "cuTensorMapEncodeTiled entry point not available");
  auto mk = [&](CUtensorMap* map, const void* base, long rows, long pitch, int box_rows) -> int {
    const cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)pitch * sizeof(__half)};
    const cuuint32_t box[2] = {(cuuint32_t)kGmBK, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) IADMM_FAIL(IADMM_ECUDA, "tc_gemm: cuTensorMapEncodeTiled failed (%d)", (int)r);
    return IADMM_OK;
  };
  CUtensorMap ma_hi, ma_lo, mb_hi, mb_lo;
  int rc;
  int num_sms = 0;
  if ((rc = device_sm_count(&num_sms))) return rc;
  // CTA pairs (256 x 256 tiles) when the tile halves are whole 8-row groups of B and there are two SMs; development switch
  // IADMM_GEMM_PAIR=0 keeps the single-CTA kernel
  const char* sw = dev_env("IADMM_GEMM_PAIR");
  const bool pair = num_sms >= 2 && !(sw && sw[0] == '0') && (N % 16 == 0);
  if ((rc = mk(&ma_hi, A_hi, M, lda, kTcBM)) || (rc = mk(&ma_lo, A_lo, M, lda, kTcBM)) ||
      (rc = mk(&mb_hi, B_hi, N, ldb, pair ? kGpBoxRows : kGmBN)) || (rc = mk(&mb_lo, B_lo, N, ldb, pair ? kGpBoxRows : kGmBN)))
    return rc;
  GemmParams P;
  if (K < 1 || splits < 1 || (splits > 1 && (!part || (M * ldc) % 4 != 0))) IADMM_FAIL(IADMM_ESHAPE, "tc_gemm: bad split-K arguments");
  P.n_tiles = (int)((N + kGmBN - 1) / kGmBN);
  P.k_blocks = (int)((K + kGmBK - 1) / kGmBK);
  P.kb_per_split = (P.k_blocks + splits - 1) / splits;
  // Only splits that cover K blocks are launched: when the factor does not divide the K blocks evenly the trailing splits
  // can be left with none (125 blocks in 15 splits of 9 cover 14 splits), and such a work unit would store an accumulator
  // that no MMA of this launch wrote.
  splits = (P.k_blocks + P.kb_per_split - 1) / P.kb_per_split;
  P.splits = splits;
  P.C = (splits > 1) ? part : C; P.scale = scale; P.M = M; P.N = N; P.K = K; P.ldc = ldc;
  P.prod_mask = prod_mask | 4;
  const int tile_rows = pair ? 2 * kTcBM : kTcBM;
  P.num_tiles = ((M + tile_rows - 1) / tile_rows) * P.n_tiles;
  static PerDeviceOnce attr, attr_pair;
  const long units = P.num_tiles * splits;
  if (pair) {
    if ((rc = ensure_dyn_smem(tc_gemm_nt_pair_kernel, 220 * 1024, &attr_pair))) return rc;
    const size_t smem = 1024 + (size_t)kGpStages * kGpStageBytes + (2 * kGpStages + 4) * sizeof(uint64_t) + 16;
    long clusters = num_sms / 2;
    if (units < clusters) clusters = units;
    tc_gemm_nt_pair_kernel<<<(unsigned)(2 * clusters), kGmThreads, smem, st>>>(ma_hi, ma_lo, mb_hi, mb_lo, P);
    IADMM_LAUNCH_CHECK("tc_gemm_nt_pair_kernel");
  } else {
    if ((rc = ensure_dyn_smem(tc_gemm_nt_kernel, 220 * 1024, &attr))) return rc;
    const size_t smem = 1024 + (size_t)kGmStages * kGmStageBytes + (2 * kGmStages + 4) * sizeof(uint64_t) + 16;
    const long grid = units < num_sms ? units : num_sms;
    tc_gemm_nt_kernel<<<(unsigned)grid, kGmThreads, smem, st>>>(ma_hi, ma_lo, mb_hi, mb_lo, P);
    IADMM_LAUNCH_CHECK("tc_gemm_nt_kernel");
  }
  if (splits > 1) {
    const size_t count4 = (size_t)(M * ldc) / 4;
    splitk_reduce_kernel<<<(unsigned)((count4 + 255) / 256), 256, 0, st>>>(reinterpret_cast<const float4*>(part),
                                                                           reinterpret_cast<float4*>(C), count4, splits);
    IADMM_LAUNCH_CHECK("splitk_reduce_kernel");
  }
  return IADMM_OK;
}

// ------------------------------------------------------------------------------------------------
// operand preparation
// ------------------------------------------------------------------------------------------------
// scales[0] = s_X = 2^(12 - ilogb(max|X|)) ; scales[1] = 1/(s_X * other[0]) ; scales[2] = 1/(s_X * 2^14)
__global__ void gemm_scales_kernel(const float* __restrict__ absmax, const float* __restrict__ other, float* __restrict__ scales) {
  const float mx = absmax[0];
  const float s = (mx > 0.f && isfinite(mx)) ? exp2f((float)(12 - ilogbf(mx))) : 1.f;
  scales[0] = s;
  scales[1] = 1.0f / (s * other[0]);
  scales[2] = 1.0f / (s * (float)(1 << kHShift));
}

__global__ void __launch_bounds__(256) absmax_kernel(const float* __restrict__ X, size_t count, float* __restrict__ out) {
  float mx = 0.f;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x) {
    const float v = fabsf(X[i]);
    if (isfinite(v)) mx = fmaxf(mx, v);
  }
  mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<int*>(out), __float_as_int(mx));
}

// X fp32 [R][Cc] -> hi/lo fp16 [R][Cc] of X * scale   (scale from device memory, or fixed 2^14 when NULL)
__global__ void __launch_bounds__(256) split_rows_kernel(const float* __restrict__ X, size_t count, const float* __restrict__ scale,
                                                         __half* __restrict__ hi, __half* __restrict__ lo) {
  const float s = scale ? scale[0] : (float)(1 << kHShift);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x) {
    const float v = X[i] * s;
    const __half a = __float2half_rn(v);
    hi[i] = a;
    lo[i] = __float2half_rn(v - __half2float(a));
  }
}

// X fp32 [R][Cc] -> hi/lo fp16 [Cc][Rp] (transposed, Rp >= R pitch; padding columns must be pre-zeroed)
__global__ void __launch_bounds__(256) split_transpose_kernel(const float* __restrict__ X, long R, long Cc, long Rp,
                                                              const float* __restrict__ scale, __half* __restrict__ hi,
                                                              __half* __restrict__ lo) {
  __shared__ float tile[32][33];
  const float s = scale ? scale[0] : (float)(1 << kHShift);
  const long r0 = (long)blockIdx.y * 32, c0 = (long)blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;     // 32 x 8
  for (int j = ty; j < 32; j += 8) {
    const long r = r0 + j, c = c0 + tx;
    tile[j][tx] = (r < R && c < Cc) ? X[r * Cc + c] * s : 0.f;
  }
  __syncthreads();
  for (int j = ty; j < 32; j += 8) {
    const long c = c0 + j, r = r0 + tx;
    if (c < Cc && r < R) {
      const float v = tile[tx][j];
      const __half a = __float2half_rn(v);
      hi[c * Rp + r] = a;
      lo[c * Rp + r] = __float2half_rn(v - __half2float(a));
    }
  }
}

// One read of X fp32 [R][Cc] -> fp16 hi/lo of X * scale both row-major [R][Cc] (hi/lo, may be NULL) and transposed
// [Cc][Rp] (thi/tlo; Rp even, padding columns pre-zeroed).  64 x 64 tiles: every global access is a full 128-byte
// (fp16 pairs) or 256-byte (fp32 pairs) warp request.
__global__ void __launch_bounds__(256) split_both_kernel(const float* __restrict__ X, long R, long Cc, long Rp,
                                                         const float* __restrict__ scale, __half* __restrict__ hi,
                                                         __half* __restrict__ lo, __half* __restrict__ thi,
                                                         __half* __restrict__ tlo) {
  __shared__ float tile[64][65];
  const float s = scale ? scale[0] : (float)(1 << kHShift);
  const long r0 = (long)blockIdx.y * 64, c0 = (long)blockIdx.x * 64;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool cvec = (Cc % 2 == 0);
  for (int j = warp; j < 64; j += 8) {
    const long r = r0 + j, c = c0 + 2 * lane;
    float v0 = 0.f, v1 = 0.f;
    if (r < R) {
      if (cvec && c + 1 < Cc) { const float2 t = *reinterpret_cast<const float2*>(X + r * Cc + c); v0 = t.x * s; v1 = t.y * s; }
      else { if (c < Cc) v0 = X[r * Cc + c] * s; if (c + 1 < Cc) v1 = X[r * Cc + c + 1] * s; }
    }
    tile[j][2 * lane] = v0; tile[j][2 * lane + 1] = v1;
    if (hi && r < R) {
      const __half2 a = __floats2half2_rn(v0, v1);
      const float2 back = __half22float2(a);
      const __half2 l = __floats2half2_rn(v0 - back.x, v1 - back.y);
      if (cvec && c + 1 < Cc) {
        *reinterpret_cast<__half2*>(hi + r * Cc + c) = a;
        *reinterpret_cast<__half2*>(lo + r * Cc + c) = l;
      } else {
        if (c < Cc) { hi[r * Cc + c] = __low2half(a); lo[r * Cc + c] = __low2half(l); }
        if (c + 1 < Cc) { hi[r * Cc + c + 1] = __high2half(a); lo[r * Cc + c + 1] = __high2half(l); }
      }
    }
  }
  __syncthreads();
  for (int j = warp; j < 64; j += 8) {
    const long c = c0 + j, r = r0 + 2 * lane;
    if (c < Cc && r < R) {
      const float v0 = tile[2 * lane][j], v1 = (r + 1 < R) ? tile[2 * lane + 1][j] : 0.f;
      const __half2 a = __floats2half2_rn(v0, v1);
      const float2 back = __half22float2(a);
      const __half2 l = __floats2half2_rn(v0 - back.x, v1 - back.y);
      if (r + 1 < Rp) {                      // Rp is even: the pair never crosses the pitch
        *reinterpret_cast<__half2*>(thi + c * Rp + r) = a;
        *reinterpret_cast<__half2*>(tlo + c * Rp + r) = l;
      } else {
        thi[c * Rp + r] = __low2half(a); tlo[c * Rp + r] = __low2half(l);
      }
    }
  }
}

int launch_split_both(const float* X, long R, long Cc, long Rp, const float* scale, __half* hi, __half* lo, __half* thi, __half* tlo,
                      cudaStream_t st) {
  const dim3 grid((unsigned)((Cc + 63) / 64), (unsigned)((R + 63) / 64));
  split_both_kernel<<<grid, 256, 0, st>>>(X, R, Cc, Rp, scale, hi, lo, thi, tlo);
  IADMM_LAUNCH_CHECK("split_both_kernel");
  return IADMM_OK;
}

int launch_absmax(const float* X, size_t count, float* out, cudaStream_t st) {
  IADMM_CUDA(cudaMemsetAsync(out, 0, sizeof(float), st));
  const size_t blocks = (count + 255) / 256;
  absmax_kernel<<<(unsigned)(blocks > 1184 ? 1184 : blocks), 256, 0, st>>>(X, count, out);
  IADMM_LAUNCH_CHECK("absmax_kernel");
  return IADMM_OK;
}
int launch_gemm_scales(const float* absmax, const float* other, float* scales, cudaStream_t st) {
  gemm_scales_kernel<<<1, 1, 0, st>>>(absmax, other, scales);
  IADMM_LAUNCH_CHECK("gemm_scales_kernel");
  return IADMM_OK;
}
int launch_split_rows(const float* X, size_t count, const float* scale, __half* hi, __half* lo, cudaStream_t st) {
  const size_t blocks = (count + 255) / 256;
  split_rows_kernel<<<(unsigned)(blocks > 148 * 16 ? 148 * 16 : blocks), 256, 0, st>>>(X, count, scale, hi, lo);
  IADMM_LAUNCH_CHECK("split_rows_kernel");
  return IADMM_OK;
}
int launch_split_transpose(const float* X, long R, long Cc, long Rp, const float* scale, __half* hi, __half* lo, cudaStream_t st) {
  const dim3 grid((unsigned)((Cc + 31) / 32), (unsigned)((R + 31) / 32));
  split_transpose_kernel<<<grid, 256, 0, st>>>(X, R, Cc, Rp, scale, hi, lo);
  IADMM_LAUNCH_CHECK("split_transpose_kernel");
  return IADMM_OK;
}

}  // namespace iadmm

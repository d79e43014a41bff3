// Stage II ("feasibility restoration") linear algebra: batched dense LU with partial pivoting and the
// triangular solves, hand-written.
//
// Reference: models/lu.py:28-35 -- `torch.lu(A_tild, pivot=True)` once, then `torch.lu_solve(b_tild, lu, piv)` in
// every Stage-II iteration (main.py:1035-1115), i.e. LAPACK getrf/getrs semantics on the dense KKT matrix
// K = [[Q + sigma I, A0^T], [A0, -diag(1/rho)]] of every instance ([B, N, N], N = n + m, row-major).
//
// Factorisation: right-looking, 16-column panels.
//   lu_panel_kernel   one CTA (1024 threads) per instance keeps the whole panel (N-k0 rows x 16 columns) in
//                     REGISTERS, one or more rows per thread: per column a block-wide arg-max (first maximum,
//                     like LAPACK's isamax), the pivot row broadcast through shared memory, a predicated
//                     register swap and the rank-1 update of the remaining panel columns.
//   lu_swap_kernel    applies the panel's 16 row interchanges to the columns outside the panel.
//   lu_trsm_kernel    U12 = L11^-1 A12 (one thread per column, L11 in shared memory).
//   lu_update_kernel  A22 -= L21 U12 (rank-16 update, memory bound: one read+write of the trailing matrix).
// Solve: lu_perm_kernel turns the pivot sequence into a permutation once; lu_solve_kernel (one CTA per instance,
// right-hand side in shared memory) runs left-looking forward and backward substitution in 32-row blocks: the
// rows of L and U are contiguous, so every row does ONE coalesced dot product with the already known part of the
// solution, then the 32x32 diagonal block is solved by a single warp from shared memory.
#include "common.cuh"
#include "tc_ptx.cuh"

namespace iadmm {

constexpr int kLuNb = 16;           // panel width
constexpr int kLuThreads = 1024;    // panel kernel threads
constexpr int kLuMaxSlots = 4;      // rows per thread held in registers -> N - k0 <= 4096

template <int SLOTS>
__global__ void __launch_bounds__(kLuThreads, 1)
lu_panel_kernel(float* __restrict__ Aall, int* __restrict__ piv_all, int* __restrict__ info, int N, int k0) {
  __shared__ float s_val[32];
  __shared__ int   s_idx[32];
  __shared__ float s_prow[kLuNb], s_orow[kLuNb];
  __shared__ int   s_piv;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float* A = Aall + (size_t)b * N * N;
  int* piv = piv_all + (size_t)b * N;
  const int kb = min(kLuNb, N - k0);

  float a[SLOTS][kLuNb];
  int   rowid[SLOTS];
#pragma unroll
  for (int s = 0; s < SLOTS; ++s) {
    const int r = k0 + tid + s * kLuThreads;
    rowid[s] = r;
#pragma unroll
    for (int c = 0; c < kLuNb; ++c) a[s][c] = (r < N && c < kb) ? A[(size_t)r * N + k0 + c] : 0.f;
  }

#pragma unroll
  for (int j = 0; j < kLuNb; ++j) {
    if (j < kb) {                                    // uniform
      const int prow_id = k0 + j;
      // ---- pivot search: first row with the largest |a[r][j]|, r >= k0 + j
      float best = -1.f; int bidx = 0x7fffffff;
#pragma unroll
      for (int s = 0; s < SLOTS; ++s) {
        if (rowid[s] >= prow_id && rowid[s] < N) {
          const float v = fabsf(a[s][j]);
          if (v > best || (v == best && rowid[s] < bidx)) { best = v; bidx = rowid[s]; }
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(kFullMask, best, o);
        const int   oi = __shfl_xor_sync(kFullMask, bidx, o);
        if (ov > best || (ov == best && oi < bidx)) { best = ov; bidx = oi; }
      }
      if (lane == 0) { s_val[warp] = best; s_idx[warp] = bidx; }
      __syncthreads();
      if (warp == 0) {
        best = s_val[lane]; bidx = s_idx[lane];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const float ov = __shfl_xor_sync(kFullMask, best, o);
          const int   oi = __shfl_xor_sync(kFullMask, bidx, o);
          if (ov > best || (ov == best && oi < bidx)) { best = ov; bidx = oi; }
        }
        if (lane == 0) {
          s_piv = bidx;
          piv[prow_id] = bidx;
          if (best == 0.f && info) atomicCAS(info + b, 0, prow_id + 1);   // exactly singular (LAPACK info > 0)
        }
      }
      __syncthreads();
      const int p = s_piv;
      // ---- publish the pivot row and the row it replaces
#pragma unroll
      for (int s = 0; s < SLOTS; ++s) {
        if (rowid[s] == p) {
#pragma unroll
          for (int c = 0; c < kLuNb; ++c) s_prow[c] = a[s][c];
        }
        if (rowid[s] == prow_id) {
#pragma unroll
          for (int c = 0; c < kLuNb; ++c) s_orow[c] = a[s][c];
        }
      }
      __syncthreads();
      // ---- interchange (registers) and eliminate below the pivot
      const float pv = s_prow[j];
      const float rinv = (pv != 0.f) ? 1.0f / pv : 0.f;
#pragma unroll
      for (int s = 0; s < SLOTS; ++s) {
        if (p != prow_id) {
          if (rowid[s] == p) {
#pragma unroll
            for (int c = 0; c < kLuNb; ++c) a[s][c] = s_orow[c];
          } else if (rowid[s] == prow_id) {
#pragma unroll
            for (int c = 0; c < kLuNb; ++c) a[s][c] = s_prow[c];
          }
        }
        if (rowid[s] > prow_id && rowid[s] < N) {
          const float l = a[s][j] * rinv;
          a[s][j] = l;
#pragma unroll
          for (int c = j + 1; c < kLuNb; ++c) a[s][c] = fmaf(-l, s_prow[c], a[s][c]);
        }
      }
      __syncthreads();                               // s_prow / s_orow / s_piv are reused by the next column
    }
  }
#pragma unroll
  for (int s = 0; s < SLOTS; ++s) {
    const int r = rowid[s];
    if (r < N) {
#pragma unroll
      for (int c = 0; c < kLuNb; ++c)
        if (c < kb) A[(size_t)r * N + k0 + c] = a[s][c];
    }
  }
}

// apply the interchanges of panel [k0, k0+kb) to the columns outside the panel.  grid (ceil(N/256), B)
__global__ void __launch_bounds__(256) lu_swap_kernel(float* __restrict__ Aall, const int* __restrict__ piv_all, int N, int k0,
                                                      int kb) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= N || (c >= k0 && c < k0 + kb)) return;
  float* A = Aall + (size_t)blockIdx.y * N * N;
  const int* piv = piv_all + (size_t)blockIdx.y * N;
  for (int j = 0; j < kb; ++j) {
    const int r = k0 + j, p = piv[r];
    if (p != r) {
      const float t = A[(size_t)r * N + c];
      A[(size_t)r * N + c] = A[(size_t)p * N + c];
      A[(size_t)p * N + c] = t;
    }
  }
}

// U12 = L11^-1 A12 for the columns right of the panel.  grid (ceil((N-k0-kb)/256), B)
__global__ void __launch_bounds__(256) lu_trsm_kernel(float* __restrict__ Aall, int N, int k0, int kb) {
  __shared__ float L11[kLuNb][kLuNb + 1];
  float* A = Aall + (size_t)blockIdx.y * N * N;
  for (int i = threadIdx.x; i < kLuNb * kLuNb; i += blockDim.x) {
    const int r = i / kLuNb, c = i % kLuNb;
    L11[r][c] = (r < kb && c < kb) ? A[(size_t)(k0 + r) * N + k0 + c] : 0.f;
  }
  __syncthreads();
  const int c = k0 + kb + blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= N) return;
  float u[kLuNb];
#pragma unroll
  for (int i = 0; i < kLuNb; ++i) {
    if (i < kb) {
      float v = A[(size_t)(k0 + i) * N + c];
#pragma unroll
      for (int t = 0; t < kLuNb; ++t)
        if (t < i) v = fmaf(-L11[i][t], u[t], v);
      u[i] = v;
      A[(size_t)(k0 + i) * N + c] = v;
    } else {
      u[i] = 0.f;
    }
  }
}

// A22 -= L21 U12.  block = 256 columns x 32 rows; grid (ceil(cols/256), ceil(rows/32), B)
__global__ void __launch_bounds__(256) lu_update_kernel(float* __restrict__ Aall, int N, int k0, int kb) {
  __shared__ float L21[32][kLuNb + 1];
  float* A = Aall + (size_t)blockIdx.z * N * N;
  const int r0 = k0 + kb + blockIdx.y * 32;
  for (int i = threadIdx.x; i < 32 * kLuNb; i += blockDim.x) {
    const int r = i / kLuNb, t = i % kLuNb;
    L21[r][t] = (r0 + r < N && t < kb) ? A[(size_t)(r0 + r) * N + k0 + t] : 0.f;
  }
  __syncthreads();
  const int c = k0 + kb + blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= N) return;
  float u[kLuNb];
#pragma unroll
  for (int t = 0; t < kLuNb; ++t) u[t] = (t < kb) ? A[(size_t)(k0 + t) * N + c] : 0.f;
#pragma unroll 4
  for (int r = 0; r < 32; ++r) {
    if (r0 + r < N) {
      float v = A[(size_t)(r0 + r) * N + c];
#pragma unroll
      for (int t = 0; t < kLuNb; ++t) v = fmaf(-L21[r][t], u[t], v);
      A[(size_t)(r0 + r) * N + c] = v;
    }
  }
}

// pivot sequence -> permutation (row i of P*K is row perm[i] of K).  One CTA per instance, sequential in smem.
__global__ void __launch_bounds__(256) lu_perm_kernel(const int* __restrict__ piv_all, int* __restrict__ perm_all, int N) {
  extern __shared__ int s_perm[];
  const int* piv = piv_all + (size_t)blockIdx.x * N;
  for (int i = threadIdx.x; i < N; i += blockDim.x) s_perm[i] = i;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 0; i < N; ++i) {
      const int p = piv[i];
      if (p != i) { const int t = s_perm[i]; s_perm[i] = s_perm[p]; s_perm[p] = t; }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < N; i += blockDim.x) perm_all[(size_t)blockIdx.x * N + i] = s_perm[i];
}

// x = U^-1 L^-1 P b.  One CTA (512 threads) per instance; dynamic smem: x[N] + diag[32][33]
constexpr int kLuSolveThreads = 512;
__global__ void __launch_bounds__(kLuSolveThreads) lu_solve_kernel(const float* __restrict__ LUall, const int* __restrict__ perm_all,
                                                                   float* __restrict__ rhs_all, int N) {
  extern __shared__ float s_mem[];
  float* x = s_mem;
  float (*diag)[33] = reinterpret_cast<float (*)[33]>(s_mem + ((N + 31) / 32) * 32);
  const float* LU = LUall + (size_t)blockIdx.x * N * N;
  const int* perm = perm_all + (size_t)blockIdx.x * N;
  float* rhs = rhs_all + (size_t)blockIdx.x * N;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int kWarps = kLuSolveThreads / 32;
  for (int i = tid; i < N; i += kLuSolveThreads) x[i] = rhs[perm[i]];
  __syncthreads();
  const int nblk = (N + 31) / 32;
  // ---- forward substitution, unit lower triangle
  for (int blk = 0; blk < nblk; ++blk) {
    const int r0 = blk * 32;
    for (int rr = warp; rr < 32; rr += kWarps) {        // rows of this block: dot with the known part x[0, r0)
      const int r = r0 + rr;
      if (r < N) {
        float acc = 0.f;
        const float* row = LU + (size_t)r * N;
        for (int c = lane; c < r0; c += 32) acc = fmaf(row[c], x[c], acc);
        acc = warp_sum(acc);
        if (lane == 0) x[r] -= acc;
        const int c = r0 + lane;                         // and stage the diagonal block
        diag[rr][lane] = (c < N) ? row[c] : 0.f;
      }
    }
    __syncthreads();
    if (warp == 0) {
      float xv = (r0 + lane < N) ? x[r0 + lane] : 0.f;
      for (int i = 0; i < 32; ++i) {
        const float xi = __shfl_sync(kFullMask, xv, i);
        if (lane > i) xv = fmaf(-diag[lane][i], xi, xv);
      }
      if (r0 + lane < N) x[r0 + lane] = xv;
    }
    __syncthreads();
  }
  // ---- backward substitution, upper triangle
  for (int blk = nblk - 1; blk >= 0; --blk) {
    const int r0 = blk * 32;
    const int c_hi = r0 + 32;                            // columns >= c_hi are known
    for (int rr = warp; rr < 32; rr += kWarps) {
      const int r = r0 + rr;
      if (r < N) {
        float acc = 0.f;
        const float* row = LU + (size_t)r * N;
        for (int c = c_hi + lane; c < N; c += 32) acc = fmaf(row[c], x[c], acc);
        acc = warp_sum(acc);
        if (lane == 0) x[r] -= acc;
        const int c = r0 + lane;
        diag[rr][lane] = (c < N) ? row[c] : 0.f;
      }
    }
    __syncthreads();
    if (warp == 0) {
      float xv = (r0 + lane < N) ? x[r0 + lane] : 0.f;
      for (int i = 31; i >= 0; --i) {
        if (r0 + i < N) {
          float xi = 0.f;
          if (lane == i) { xv = xv / diag[i][i]; }
          xi = __shfl_sync(kFullMask, xv, i);
          if (lane < i) xv = fmaf(-diag[lane][i], xi, xv);
        }
      }
      if (r0 + lane < N) x[r0 + lane] = xv;
    }
    __syncthreads();
  }
  for (int i = tid; i < N; i += kLuSolveThreads) rhs[i] = x[i];
}

// ================================================================================================
// Blocked factorisation for N up to 32768 (iadmm_lu_factor_blocked): right-looking, outer blocks of kLuBlkNb columns.
//   per outer block [k0, k0+nb):
//     for every 16-column sub-panel [j0, j0+kb):
//       lu_panel_cluster_kernel   rows j0..N-1 on a cluster of C CTAs, 4096 rows per CTA; per column a CTA-local arg-max,
//                                 the candidates exchanged through distributed shared memory, the pivot row and the row
//                                 it replaces written into every CTA, then the register swap and rank-1 update
//       lu_swap_band_kernel       the sub-panel's interchanges on the other columns of the outer block
//       lu_trsm_nb_kernel<16>     U of the sub-panel rows on the block columns right of it
//       lu_update_band_kernel     rank-16 update of the block columns right of it (a band of < 128 columns, L2 resident)
//     lu_swap_kernel              the block's interchanges on every column outside it (LAPACK's laswp, once per block)
//     lu_trsm_nb_kernel<128>      U12 = L11^-1 A12
//     lu_split_l/_ut_kernel       L21 and U12^T as tf32 hi/lo images, K-major, in the workspace
//     lu_tf32_update_kernel       A22 -= L21 U12 on the tensor cores: hi*hi + hi*lo + lo*hi accumulated in fp32 in TMEM
// ================================================================================================
constexpr int kLuBlkNb = 128;           // outer block width = K of the trailing update
constexpr int kLuSlice = kLuThreads * kLuMaxSlots;   // rows per CTA of the cluster panel
constexpr int kLuMaxCluster = 8;        // portable cluster size -> N <= 32768
constexpr int kLuBlkMaxN = kLuSlice * kLuMaxCluster;

__device__ __forceinline__ void st_cluster_f32(uint32_t addr, float v) {
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ void st_cluster_s32(uint32_t addr, int v) {
  asm volatile("st.shared::cluster.s32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// One 16-column sub-panel, rows j0..N-1, on a cluster of `csize` CTAs (grid (csize, B)).  CTA `rank` owns rows
// j0 + rank * kLuSlice + tid + s * 1024 for s < RS + SS: slots s < RS live in registers, the others in dynamic shared
// memory ([SS][16][1024], one column per bank row), because a 4096 x 16 panel slice is the whole register file (the
// 4-slot register-only lu_panel_kernel spills).  A 4096-row slice runs as RS = 1, SS = 3 (192 KB of shared memory).
// Per column: two barriers (the cluster barrier when csize > 1): one after the arg-max candidates are exchanged, one
// after the pivot row and the row it replaces are published.  Every CTA reduces the candidates in rank order with
// isamax's rule (largest magnitude, then smallest row), so all CTAs agree on the pivot.
template <int RS, int SS>
__global__ void __launch_bounds__(kLuThreads, 1)
lu_panel_cluster_kernel(float* __restrict__ Aall, int* __restrict__ piv_all, int* __restrict__ info, int N, int j0, int kb,
                        int csize) {
  constexpr int SLOTS = RS + SS;
  extern __shared__ float s_slot[];                  // [SS][kLuNb][kLuThreads]
  __shared__ float s_val[32];
  __shared__ int   s_idx[32];
  __shared__ float s_prow[kLuNb], s_orow[kLuNb];
  __shared__ float s_cval[kLuMaxCluster];
  __shared__ int   s_cidx[kLuMaxCluster];
  const int b = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t rank = cluster_ctarank();
  float* A = Aall + (size_t)b * N * N;
  int* piv = piv_all + (size_t)b * N;

  float a[RS > 0 ? RS : 1][kLuNb];
  int rowid[SLOTS];
#define LU_SLOT(s, c) s_slot[(((s) - RS) * kLuNb + (c)) * kLuThreads + tid]
#define LU_LD(s, c) ((s) < RS ? a[(s) < RS ? (s) : 0][c] : LU_SLOT(s, c))
#define LU_ST(s, c, v)                          \
  do {                                          \
    if ((s) < RS) a[(s) < RS ? (s) : 0][c] = (v); \
    else LU_SLOT(s, c) = (v);                   \
  } while (0)
#pragma unroll
  for (int s = 0; s < SLOTS; ++s) {
    const int r = j0 + (int)rank * (SLOTS * kLuThreads) + tid + s * kLuThreads;
    rowid[s] = r;
#pragma unroll
    for (int c = 0; c < kLuNb; ++c) LU_ST(s, c, (r < N && c < kb) ? A[(size_t)r * N + j0 + c] : 0.f);
  }
  // a single CTA keeps to plain shared-memory stores and __syncthreads
  auto sync_all = [&]() {
    if (csize > 1) cluster_sync_all();
    else __syncthreads();
  };
  auto put_f32 = [&](float* local, uint32_t q, float v) {
    if (csize > 1) st_cluster_f32(map_to_cta(smem_u32(local), q), v);
    else *local = v;
  };
  auto put_s32 = [&](int* local, uint32_t q, int v) {
    if (csize > 1) st_cluster_s32(map_to_cta(smem_u32(local), q), v);
    else *local = v;
  };

#pragma unroll
  for (int j = 0; j < kLuNb; ++j) {
    if (j < kb) {                                    // uniform
      const int prow_id = j0 + j;
      float best = -1.f; int bidx = 0x7fffffff;
#pragma unroll
      for (int s = 0; s < SLOTS; ++s) {
        if (rowid[s] >= prow_id && rowid[s] < N) {
          const float v = fabsf(LU_LD(s, j));
          if (v > best || (v == best && rowid[s] < bidx)) { best = v; bidx = rowid[s]; }
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(kFullMask, best, o);
        const int   oi = __shfl_xor_sync(kFullMask, bidx, o);
        if (ov > best || (ov == best && oi < bidx)) { best = ov; bidx = oi; }
      }
      if (lane == 0) { s_val[warp] = best; s_idx[warp] = bidx; }
      __syncthreads();
      if (warp == 0) {
        best = s_val[lane]; bidx = s_idx[lane];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const float ov = __shfl_xor_sync(kFullMask, best, o);
          const int   oi = __shfl_xor_sync(kFullMask, bidx, o);
          if (ov > best || (ov == best && oi < bidx)) { best = ov; bidx = oi; }
        }
        // this CTA's candidate into slot `rank` of every CTA of the cluster
        if (lane < csize) {
          put_f32(&s_cval[rank], (uint32_t)lane, best);
          put_s32(&s_cidx[rank], (uint32_t)lane, bidx);
        }
      }
      sync_all();
      best = s_cval[0]; bidx = s_cidx[0];
      for (int q = 1; q < csize; ++q) {
        const float ov = s_cval[q];
        const int   oi = s_cidx[q];
        if (ov > best || (ov == best && oi < bidx)) { best = ov; bidx = oi; }
      }
      const int p = bidx;
      if (rank == 0 && tid == 0) {
        piv[prow_id] = p;
        if (best == 0.f && info) atomicCAS(info + b, 0, prow_id + 1);   // exactly singular (LAPACK info > 0)
      }
      // ---- the owners publish the pivot row and the row it replaces into every CTA
#pragma unroll
      for (int s = 0; s < SLOTS; ++s) {
        if (rowid[s] == p || rowid[s] == prow_id) {
          for (int q = 0; q < csize; ++q) {
#pragma unroll
            for (int c = 0; c < kLuNb; ++c) {
              const float v = LU_LD(s, c);
              if (rowid[s] == p) put_f32(&s_prow[c], (uint32_t)q, v);
              if (rowid[s] == prow_id) put_f32(&s_orow[c], (uint32_t)q, v);
            }
          }
        }
      }
      sync_all();
      // ---- interchange and eliminate below the pivot
      const float pv = s_prow[j];
      const float rinv = (pv != 0.f) ? 1.0f / pv : 0.f;
#pragma unroll
      for (int s = 0; s < SLOTS; ++s) {
        if (p != prow_id) {
          if (rowid[s] == p) {
#pragma unroll
            for (int c = 0; c < kLuNb; ++c) LU_ST(s, c, s_orow[c]);
          } else if (rowid[s] == prow_id) {
#pragma unroll
            for (int c = 0; c < kLuNb; ++c) LU_ST(s, c, s_prow[c]);
          }
        }
        if (rowid[s] > prow_id && rowid[s] < N) {
          const float l = LU_LD(s, j) * rinv;
          LU_ST(s, j, l);
#pragma unroll
          for (int c = j + 1; c < kLuNb; ++c) LU_ST(s, c, fmaf(-l, s_prow[c], LU_LD(s, c)));
        }
      }
      // s_val/s_idx, s_cval/s_cidx and s_prow/s_orow are rewritten only after the next column's first barrier
    }
  }
#pragma unroll
  for (int s = 0; s < SLOTS; ++s) {
    const int r = rowid[s];
    if (r < N) {
#pragma unroll
      for (int c = 0; c < kLuNb; ++c)
        if (c < kb) A[(size_t)r * N + j0 + c] = LU_LD(s, c);
    }
  }
#undef LU_SLOT
#undef LU_LD
#undef LU_ST
  if (csize > 1) cluster_sync_all();                 // no CTA exits while a peer may still write into its shared memory
}

// interchanges of sub-panel [j0, j0+kb) on the columns [c_begin, c_end) outside it.  grid (ceil((c_end-c_begin)/128), B)
__global__ void __launch_bounds__(128) lu_swap_band_kernel(float* __restrict__ Aall, const int* __restrict__ piv_all, int N, int j0,
                                                           int kb, int c_begin, int c_end) {
  const int c = c_begin + blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= c_end || (c >= j0 && c < j0 + kb)) return;
  float* A = Aall + (size_t)blockIdx.y * N * N;
  const int* piv = piv_all + (size_t)blockIdx.y * N;
  for (int j = 0; j < kb; ++j) {
    const int r = j0 + j, p = piv[r];
    if (p != r) {
      const float t = A[(size_t)r * N + c];
      A[(size_t)r * N + c] = A[(size_t)p * N + c];
      A[(size_t)p * N + c] = t;
    }
  }
}

// U = L11^-1 A for rows [k0, k0+kb) (kb <= W) and columns [c_begin, c_end).  The strictly lower part of the W x W unit
// lower L11 sits packed in shared memory; each thread solves one column in fp32, 16 rows at a time in registers, the
// finished rows of its column kept in dynamic shared memory ([W][128], W * 512 bytes).  Every row subtracts its terms in
// ascending column order, as lu_trsm_kernel does.  grid (ceil((c_end-c_begin)/128), B), 128 threads
__host__ __device__ constexpr int lu_tri(int i, int t) { return i * (i - 1) / 2 + t; }
constexpr int kLuTrsmThreads = 128;
template <int W>
__global__ void __launch_bounds__(kLuTrsmThreads) lu_trsm_nb_kernel(float* __restrict__ Aall, int N, int k0, int kb, int c_begin,
                                                                    int c_end) {
  __shared__ float L11[lu_tri(W, 0)];
  extern __shared__ float s_u[];
  float* A = Aall + (size_t)blockIdx.y * N * N;
  const int tid = threadIdx.x;
  for (int i = tid; i < W * W; i += kLuTrsmThreads) {
    const int r = i / W, c = i % W;
    if (c < r) L11[lu_tri(r, c)] = (r < kb) ? A[(size_t)(k0 + r) * N + k0 + c] : 0.f;
  }
  __syncthreads();
  const int c = c_begin + blockIdx.x * kLuTrsmThreads + tid;
  if (c >= c_end) return;
#pragma unroll 1
  for (int i0 = 0; i0 < kb; i0 += kLuNb) {
    float v[kLuNb];
#pragma unroll
    for (int i = 0; i < kLuNb; ++i) v[i] = (i0 + i < kb) ? A[(size_t)(k0 + i0 + i) * N + c] : 0.f;
#pragma unroll 1
    for (int t = 0; t < i0; ++t) {                   // rows solved in earlier chunks
      const float ut = s_u[t * kLuTrsmThreads + tid];
#pragma unroll
      for (int i = 0; i < kLuNb; ++i) v[i] = fmaf(-L11[lu_tri(i0 + i, t)], ut, v[i]);
    }
#pragma unroll
    for (int i = 0; i < kLuNb; ++i) {
#pragma unroll
      for (int t = 0; t < i; ++t) v[i] = fmaf(-L11[lu_tri(i0 + i, i0 + t)], v[t], v[i]);
      if (i0 + i < kb) {
        s_u[(i0 + i) * kLuTrsmThreads + tid] = v[i];
        A[(size_t)(k0 + i0 + i) * N + c] = v[i];
      }
    }
  }
}

// rows [j0+kb, N) x columns [j0+kb, c_end) -= L21 U12 for the sub-panel [j0, j0+kb).  block = 128 columns x 32 rows;
// grid (ceil((c_end-j0-kb)/128), ceil((N-j0-kb)/32), B)
__global__ void __launch_bounds__(128) lu_update_band_kernel(float* __restrict__ Aall, int N, int j0, int kb, int c_end) {
  __shared__ float L21[32][kLuNb + 1];
  float* A = Aall + (size_t)blockIdx.z * N * N;
  const int r0 = j0 + kb + blockIdx.y * 32;
  for (int i = threadIdx.x; i < 32 * kLuNb; i += blockDim.x) {
    const int r = i / kLuNb, t = i % kLuNb;
    L21[r][t] = (r0 + r < N && t < kb) ? A[(size_t)(r0 + r) * N + j0 + t] : 0.f;
  }
  __syncthreads();
  const int c = j0 + kb + blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= c_end) return;
  float u[kLuNb];
#pragma unroll
  for (int t = 0; t < kLuNb; ++t) u[t] = (t < kb) ? A[(size_t)(j0 + t) * N + c] : 0.f;
#pragma unroll 4
  for (int r = 0; r < 32; ++r) {
    if (r0 + r < N) {
      float v = A[(size_t)(r0 + r) * N + c];
#pragma unroll
      for (int t = 0; t < kLuNb; ++t) v = fmaf(-L21[r][t], u[t], v);
      A[(size_t)(r0 + r) * N + c] = v;
    }
  }
}

// tf32 split: hi = x rounded to tf32 (to nearest, the low 13 mantissa bits zero), lo = tf32(x - hi).  Rounding hi
// rather than truncating it halves |lo| <= 2^-11 |x|, so the dropped lo*lo product stays below 2^-22 relative.
__device__ __forceinline__ float tf32_rna(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
__device__ __forceinline__ void tf32_split(float x, float& hi, float& lo) {
  hi = tf32_rna(x);
  lo = tf32_rna(x - hi);
}

// L21 = rows [r0, r0+M) x columns [k0, k0+kb) -> hi/lo [B][N][kLuBlkNb] (K-major rows; K columns >= kb are zero).
// grid (ceil(M*kLuBlkNb/256), B)
__global__ void __launch_bounds__(256) lu_split_l_kernel(const float* __restrict__ Aall, int N, int k0, int kb, int M,
                                                         float* __restrict__ hi, float* __restrict__ lo) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)M * kLuBlkNb) return;
  const int r = (int)(i / kLuBlkNb), k = (int)(i % kLuBlkNb);
  const float* A = Aall + (size_t)blockIdx.y * N * N;
  const float x = (k < kb) ? A[(size_t)(k0 + kb + r) * N + k0 + k] : 0.f;
  float h, l;
  tf32_split(x, h, l);
  const size_t o = (size_t)blockIdx.y * N * kLuBlkNb + i;
  hi[o] = h; lo[o] = l;
}

// U12^T: rows [k0, k0+kb) x columns [c0, c0+M) (c0 = k0+kb) -> hi/lo [B][N][kLuBlkNb], row c holding column c0+c.
// grid (ceil(M/32), kLuBlkNb/32, B), 32 x 8 threads
__global__ void __launch_bounds__(256) lu_split_ut_kernel(const float* __restrict__ Aall, int N, int k0, int kb, int M,
                                                          float* __restrict__ hi, float* __restrict__ lo) {
  __shared__ float tile[32][33];
  const float* A = Aall + (size_t)blockIdx.z * N * N;
  const int c_base = blockIdx.x * 32, k_base = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int j = ty; j < 32; j += 8) {
    const int k = k_base + j, c = c_base + tx;
    tile[j][tx] = (k < kb && c < M) ? A[(size_t)(k0 + k) * N + k0 + kb + c] : 0.f;
  }
  __syncthreads();
  for (int j = ty; j < 32; j += 8) {
    const int c = c_base + j, k = k_base + tx;
    if (c < M) {
      float h, l;
      tf32_split(tile[tx][j], h, l);
      const size_t o = ((size_t)blockIdx.z * N + c) * kLuBlkNb + k;
      hi[o] = h; lo[o] = l;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// A22 -= L21 U12 on CTA pairs (cta_group::2), kind::tf32.  Tile 256 x 256 per pair, K = kLuBlkNb in 32-element (128-byte,
// 128B-swizzled) stages fed by TMA from the hi/lo images (3D tensor maps {K, M, B}: rows past M read as zero).  Barrier
// protocol of tc_gemm_nt_pair_kernel (gemm_tc.cu): every CTA loads its 128 rows of L21 and its half (128 rows) of U12^T,
// the leader issues M = 256 MMAs, `full` (leader) counts both CTAs' bytes, `empty` and `tmem_full` are signalled in both
// CTAs by multicast commits, `tmem_empty` (leader) collects the epilogue warps of both.  hi*hi accumulates in TMEM columns
// [0, 256) and the two correction products in [256, 512): the tensor core's fp32 accumulation does not round to nearest,
// and a separate accumulator keeps the corrections' 32 extra accumulations per K block off the large main sum.  The
// epilogue adds the two in fp32.  With both halves of TMEM in use the accumulators are not double-buffered.  The epilogue stages each 32 x 32
// accumulator block through shared memory so that the load of A22, the subtraction and the store run along rows: every
// element of A22 has exactly one writer (no split-K), so the result does not depend on scheduling.
// ------------------------------------------------------------------------------------------------
constexpr int kLgBK = 32;                                  // tf32 elements per stage row (128 bytes)
constexpr int kLgUK = 8;                                   // UMMA K for kind::tf32
constexpr int kLgBN = 256;
constexpr int kLgOpBytes = kTcBM * kLgBK * 4;              // 16 KB: 128 rows of one operand image
constexpr int kLgStageBytes = 4 * kLgOpBytes;              // L hi, L lo, U hi, U lo
constexpr int kLgStages = 3;
constexpr int kLgEpiWarps = 8;
constexpr int kLgThreads = 32 * (2 + kLgEpiWarps);
constexpr int kLgEpiBytes = kLgEpiWarps * 32 * 33 * 4;
constexpr size_t kLgSmem = 1024 + (size_t)kLgStages * kLgStageBytes + kLgEpiBytes + (2 * kLgStages + 4) * sizeof(uint64_t) + 16;

struct LuGemmParams {
  float* A;                // [B][N][N]
  int N, r0, M;            // A22 = rows/columns [r0, r0+M)
  int tiles_m, tiles_n;    // 256-row / 256-column tiles per instance
  long units;              // B * tiles_m * tiles_n
  int k_blocks;
};

// kind::tf32 instruction descriptor: D = f32, A = B = tf32, both K-major
__device__ __forceinline__ uint32_t make_idesc_tf32(int n_cols, int m_rows) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n_cols >> 3) << 17) | ((uint32_t)(m_rows >> 4) << 24);
}
__device__ __forceinline__ void tc_mma_tf32_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kLgThreads, 1)
lu_tf32_update_kernel(const __grid_constant__ CUtensorMap map_l_hi, const __grid_constant__ CUtensorMap map_l_lo,
                      const __grid_constant__ CUtensorMap map_u_hi, const __grid_constant__ CUtensorMap map_u_lo,
                      const LuGemmParams P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  float* epi = reinterpret_cast<float*>(smem + (size_t)kLgStages * kLgStageBytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)kLgStages * kLgStageBytes + kLgEpiBytes);
  uint64_t* full_bar = bars;                         // [stages]  (leader's copy is the live one)
  uint64_t* empty_bar = bars + kLgStages;            // [stages]  both CTAs
  uint64_t* tfull_bar = bars + 2 * kLgStages;        // [2]       both CTAs
  uint64_t* tempty_bar = bars + 2 * kLgStages + 2;   // [2]       leader's copy is the live one
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kLgStages + 4);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const long tiles = (long)P.tiles_m * P.tiles_n;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_l_hi); tma_prefetch_desc(&map_l_lo); tma_prefetch_desc(&map_u_hi); tma_prefetch_desc(&map_u_lo);
    for (int s = 0; s < kLgStages; ++s) { mbar_init(smem_u32(&full_bar[s]), 1); mbar_init(smem_u32(&empty_bar[s]), 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(smem_u32(&tfull_bar[b]), 1); mbar_init(smem_u32(&tempty_bar[b]), 2 * kLgEpiWarps); }
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

  if (warp == 0) {
    // ===================== TMA producer (every CTA) =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (long unit = pair; unit < P.units; unit += num_pairs) {
        const int b = (int)(unit / tiles);
        const long t = unit - (long)b * tiles;
        const int mt = (int)(t / P.tiles_n), nt = (int)(t - (long)mt * P.tiles_n);
        const int row0 = mt * (2 * kTcBM) + (int)rank * kTcBM;          // this CTA's 128 rows of L21
        const int col0 = nt * kLgBN + (int)rank * (kLgBN / 2);           // this CTA's half of the U12^T tile
        for (int kb = 0; kb < P.k_blocks; ++kb) {
          mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1);
          const uint32_t fb_local = smem_u32(&full_bar[stage]);
          if (leader) mbar_expect_tx(fb_local, 2u * kLgStageBytes);
          const uint32_t fb = map_to_cta(fb_local, 0);
          const uint32_t sb = smem_u32(smem + (size_t)stage * kLgStageBytes);
          const int k0 = kb * kLgBK;
          tma_load_3d_pair(sb, &map_l_hi, fb, k0, row0, b);
          tma_load_3d_pair(sb + kLgOpBytes, &map_l_lo, fb, k0, row0, b);
          tma_load_3d_pair(sb + 2 * kLgOpBytes, &map_u_hi, fb, k0, col0, b);
          tma_load_3d_pair(sb + 3 * kLgOpBytes, &map_u_lo, fb, k0, col0, b);
          if (++stage == kLgStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (leader && lane == 0) {
      const uint32_t idesc = make_idesc_tf32(kLgBN, 2 * kTcBM);
      int stage = 0; uint32_t phase = 0;
      long it = 0;
      for (long unit = pair; unit < P.units; unit += num_pairs, ++it) {
        mbar_wait(smem_u32(&tempty_bar[0]), (uint32_t)(it & 1) ^ 1);   // both CTAs' epilogues drained the accumulators
        tc_fence_after();
        const uint32_t d_main = tmem_base, d_corr = tmem_base + kLgBN;
        uint32_t acc = 0;
        for (int kb = 0; kb < P.k_blocks; ++kb) {
          mbar_wait(smem_u32(&full_bar[stage]), phase);
          tc_fence_after();
          const uint32_t sb = smem_u32(smem + (size_t)stage * kLgStageBytes);
#pragma unroll
          for (int ks = 0; ks < kLgBK / kLgUK; ++ks) {
            const uint32_t koff = (uint32_t)(ks * kLgUK * 4);
            const uint64_t l_hi = make_smem_desc_sw128(sb + koff);
            const uint64_t l_lo = make_smem_desc_sw128(sb + kLgOpBytes + koff);
            const uint64_t u_hi = make_smem_desc_sw128(sb + 2 * kLgOpBytes + koff);
            const uint64_t u_lo = make_smem_desc_sw128(sb + 3 * kLgOpBytes + koff);
            tc_mma_tf32_pair(d_corr, l_lo, u_hi, idesc, acc);
            tc_mma_tf32_pair(d_corr, l_hi, u_lo, idesc, 1);
            tc_mma_tf32_pair(d_main, l_hi, u_hi, idesc, acc); acc = 1;
          }
          tc_commit_pair(smem_u32(&empty_bar[stage]), (uint16_t)3);   // frees the stage in both CTAs when the MMAs retire
          if (++stage == kLgStages) { stage = 0; phase ^= 1; }
        }
        tc_commit_pair(smem_u32(&tfull_bar[0]), (uint16_t)3);         // accumulators complete in both CTAs
      }
    }
  } else {
    // ===================== epilogue (both CTAs, own 128 rows) =====================
    const int ew = warp - 2;
    const int quarter = warp & 3;                    // TMEM lane quarter this warp may access
    const int half = (ew >= 4) ? 1 : 0;
    float (*stage_buf)[33] = reinterpret_cast<float (*)[33]>(epi + ew * 32 * 33);
    long it = 0;
    for (long unit = pair; unit < P.units; unit += num_pairs, ++it) {
      const int b = (int)(unit / tiles);
      const long t = unit - (long)b * tiles;
      const int mt = (int)(t / P.tiles_n), nt = (int)(t - (long)mt * P.tiles_n);
      const int row_base = mt * (2 * kTcBM) + (int)rank * kTcBM + quarter * 32;     // within A22
      float* A = P.A + (size_t)b * P.N * P.N + (size_t)P.r0 * P.N + P.r0;
      mbar_wait(smem_u32(&tfull_bar[0]), (uint32_t)(it & 1));
      tc_fence_after();
#pragma unroll 1
      for (int cc = 0; cc < 4; ++cc) {
        const int chunk = half * 4 + cc;
        const int col = nt * kLgBN + chunk * 32 + lane;
        uint32_t v[32];
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(chunk * 32);
        tc_ld32(taddr, v);                           // hi*hi
        tc_wait_ld();
#pragma unroll
        for (int q = 0; q < 32; ++q) stage_buf[lane][q] = __uint_as_float(v[q]);     // lane = row, q = column
        tc_ld32(taddr + kLgBN, v);                   // + the corrections
        tc_wait_ld();
#pragma unroll
        for (int q = 0; q < 32; ++q) stage_buf[lane][q] += __uint_as_float(v[q]);
        __syncwarp();
        // A22 -= the block, along rows, 16 independent row loads in flight per warp
#pragma unroll 1
        for (int r0 = 0; r0 < 32; r0 += 16) {
          float* base = A + (size_t)(row_base + r0) * P.N + col;
          float a22[16];
#pragma unroll
          for (int rr = 0; rr < 16; ++rr)
            a22[rr] = (col < P.M && row_base + r0 + rr < P.M) ? base[(size_t)rr * P.N] : 0.f;
#pragma unroll
          for (int rr = 0; rr < 16; ++rr)
            if (col < P.M && row_base + r0 + rr < P.M) base[(size_t)rr * P.N] = a22[rr] - stage_buf[r0 + rr][lane];
        }
        __syncwarp();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(map_to_cta(smem_u32(&tempty_bar[0]), 0));
    }
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

// 3D tensor map over a hi/lo image [B][N][kLuBlkNb] fp32 with M live rows per instance: box 32 K x 128 rows x 1 instance,
// 128B swizzle, rows past M read as zero
static int lu_make_map(CUtensorMap* map, const float* base, int B, int N, int M) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) IADMM_FAIL(IADMM_ECUDA, "cuTensorMapEncodeTiled entry point not available");
  const cuuint64_t dims[3] = {(cuuint64_t)kLuBlkNb, (cuuint64_t)M, (cuuint64_t)B};
  const cuuint64_t strides[2] = {(cuuint64_t)kLuBlkNb * 4, (cuuint64_t)N * kLuBlkNb * 4};
  const cuuint32_t box[3] = {(cuuint32_t)kLgBK, (cuuint32_t)kTcBM, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) IADMM_FAIL(IADMM_ECUDA, "lu_factor_blocked: cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return IADMM_OK;
}

// one 16-column sub-panel on a cluster of C = next power of two >= ceil(rows / 4096) CTAs (1 CTA: the register-only
// variants while the rows fit them)
static int lu_launch_panel(float* K, int* piv, int* info, int B, int N, int j0, int kb, cudaStream_t st) {
  const int rows = N - j0;
  int csize = 1;
  while (csize * kLuSlice < rows) csize *= 2;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)csize, (unsigned)B); cfg.blockDim = dim3(kLuThreads); cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = (unsigned)csize; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  if (csize == 1 && rows <= kLuThreads) {
    IADMM_CUDA(cudaLaunchKernelEx(&cfg, lu_panel_cluster_kernel<1, 0>, K, piv, info, N, j0, kb, csize));
  } else if (csize == 1 && rows <= 2 * kLuThreads) {
    IADMM_CUDA(cudaLaunchKernelEx(&cfg, lu_panel_cluster_kernel<2, 0>, K, piv, info, N, j0, kb, csize));
  } else {
    static PerDeviceOnce attr;
    constexpr int smem = 3 * kLuNb * kLuThreads * (int)sizeof(float);      // 192 KB: slots 1 to 3
    int rc;
    if ((rc = ensure_dyn_smem(lu_panel_cluster_kernel<1, 3>, smem, &attr))) return rc;
    cfg.dynamicSmemBytes = smem;
    IADMM_CUDA(cudaLaunchKernelEx(&cfg, lu_panel_cluster_kernel<1, 3>, K, piv, info, N, j0, kb, csize));
  }
  IADMM_LAUNCH_CHECK("lu_panel_cluster_kernel");
  return IADMM_OK;
}

static size_t lu_blocked_image_bytes(int B, int N) { return (size_t)B * N * kLuBlkNb * sizeof(float); }

}  // namespace iadmm

using namespace iadmm;

extern "C" {

int iadmm_lu_factor(float* K, int* piv, int* perm, int* info, int B, int N, void* stream) {
  if (B <= 0 || N <= 0) IADMM_FAIL(IADMM_ESHAPE, "lu_factor: B=%d N=%d", B, N);
  if (B > 65535) IADMM_FAIL(IADMM_ESHAPE, "lu_factor: batch %d > 65535", B);
  if (N > kLuThreads * kLuMaxSlots) IADMM_FAIL(IADMM_EMODE, "lu_factor: N=%d exceeds the register-resident panel limit %d", N, kLuThreads * kLuMaxSlots);
  if (!K || !piv || !perm) IADMM_FAIL(IADMM_EALIGN, "lu_factor: NULL pointer");
  int dev = 0, major = 0;
  IADMM_CUDA(cudaGetDevice(&dev));
  IADMM_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  if (major != 10) IADMM_FAIL(IADMM_EARCH, "device %d has compute capability %d.x; libiadmm_b200 needs sm_100 (B200)", dev, major);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (info) IADMM_CUDA(cudaMemsetAsync(info, 0, (size_t)B * sizeof(int), st));
  for (int k0 = 0; k0 < N; k0 += kLuNb) {
    const int kb = (N - k0 < kLuNb) ? N - k0 : kLuNb;
    const int rows = N - k0;
    if (rows <= kLuThreads)          lu_panel_kernel<1><<<B, kLuThreads, 0, st>>>(K, piv, info, N, k0);
    else if (rows <= 2 * kLuThreads) lu_panel_kernel<2><<<B, kLuThreads, 0, st>>>(K, piv, info, N, k0);
    else                             lu_panel_kernel<4><<<B, kLuThreads, 0, st>>>(K, piv, info, N, k0);
    IADMM_LAUNCH_CHECK("lu_panel_kernel");
    lu_swap_kernel<<<dim3(cdiv(N, 256), B), 256, 0, st>>>(K, piv, N, k0, kb);
    IADMM_LAUNCH_CHECK("lu_swap_kernel");
    const int rest = N - k0 - kb;
    if (rest > 0) {
      lu_trsm_kernel<<<dim3(cdiv(rest, 256), B), 256, 0, st>>>(K, N, k0, kb);
      IADMM_LAUNCH_CHECK("lu_trsm_kernel");
      lu_update_kernel<<<dim3(cdiv(rest, 256), cdiv(rest, 32), B), 256, 0, st>>>(K, N, k0, kb);
      IADMM_LAUNCH_CHECK("lu_update_kernel");
    }
  }
  lu_perm_kernel<<<B, 256, (size_t)N * sizeof(int), st>>>(piv, perm, N);
  IADMM_LAUNCH_CHECK("lu_perm_kernel");
  return IADMM_OK;
}

int iadmm_lu_solve(const float* LU, const int* perm, float* rhs, int B, int N, void* stream) {
  if (B <= 0 || N <= 0) IADMM_FAIL(IADMM_ESHAPE, "lu_solve: B=%d N=%d", B, N);
  if (!LU || !perm || !rhs) IADMM_FAIL(IADMM_EALIGN, "lu_solve: NULL pointer");
  const size_t smem = ((size_t)((N + 31) / 32) * 32 + 32 * 33) * sizeof(float);
  if (smem > 200 * 1024) IADMM_FAIL(IADMM_EMODE, "lu_solve: N=%d does not fit the shared-memory right-hand side", N);
  static PerDeviceOnce attr;
  int rc;
  if ((rc = ensure_dyn_smem(lu_solve_kernel, 200 * 1024, &attr))) return rc;
  lu_solve_kernel<<<B, kLuSolveThreads, smem, static_cast<cudaStream_t>(stream)>>>(LU, perm, rhs, N);
  IADMM_LAUNCH_CHECK("lu_solve_kernel");
  return IADMM_OK;
}

static int lu_blocked_shape(const char* who, int B, int N) {
  if (B <= 0 || N <= 0) IADMM_FAIL(IADMM_ESHAPE, "%s: B=%d N=%d", who, B, N);
  if (B > 65535) IADMM_FAIL(IADMM_ESHAPE, "%s: batch %d > 65535", who, B);
  if (N > kLuBlkMaxN) IADMM_FAIL(IADMM_EMODE, "%s: N=%d exceeds %d (%d-CTA panel clusters of %d rows)", who, N, kLuBlkMaxN,
                                 kLuMaxCluster, kLuSlice);
  return IADMM_OK;
}

int iadmm_lu_factor_blocked_workspace_bytes(int B, int N, size_t* bytes) {
  int rc;
  if ((rc = lu_blocked_shape("lu_factor_blocked_workspace_bytes", B, N))) return rc;
  if (!bytes) IADMM_FAIL(IADMM_EALIGN, "lu_factor_blocked_workspace_bytes: NULL pointer");
  *bytes = 4 * align_up(lu_blocked_image_bytes(B, N), 256) + 256;     // L21 hi/lo, U12^T hi/lo (+ alignment slack)
  return IADMM_OK;
}

int iadmm_lu_factor_blocked(float* K, int* piv, int* perm, int* info, int B, int N, void* workspace, size_t workspace_bytes,
                            void* stream) {
  int rc;
  if ((rc = lu_blocked_shape("lu_factor_blocked", B, N))) return rc;
  if (!K || !piv || !perm || !workspace) IADMM_FAIL(IADMM_EALIGN, "lu_factor_blocked: NULL pointer");
  size_t need = 0;
  if ((rc = iadmm_lu_factor_blocked_workspace_bytes(B, N, &need))) return rc;
  if (workspace_bytes < need) IADMM_FAIL(IADMM_EWORK, "lu_factor_blocked: workspace %zu bytes < %zu", workspace_bytes, need);
  if ((rc = check_device())) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t img = align_up(lu_blocked_image_bytes(B, N), 256);
  uint8_t* ws = reinterpret_cast<uint8_t*>(align_up(reinterpret_cast<uintptr_t>(workspace), 256));
  float* l_hi = reinterpret_cast<float*>(ws);
  float* l_lo = reinterpret_cast<float*>(ws + img);
  float* u_hi = reinterpret_cast<float*>(ws + 2 * img);
  float* u_lo = reinterpret_cast<float*>(ws + 3 * img);
  int num_sms = 0;
  if ((rc = device_sm_count(&num_sms))) return rc;
  static PerDeviceOnce attr_gemm, attr_perm, attr_trsm;
  if ((rc = ensure_dyn_smem(lu_tf32_update_kernel, (int)kLgSmem, &attr_gemm))) return rc;
  if ((rc = ensure_dyn_smem(lu_trsm_nb_kernel<kLuBlkNb>, kLuBlkNb * kLuTrsmThreads * (int)sizeof(float), &attr_trsm))) return rc;
  if ((rc = ensure_dyn_smem(lu_perm_kernel, kLuBlkMaxN * (int)sizeof(int), &attr_perm))) return rc;

  if (info) IADMM_CUDA(cudaMemsetAsync(info, 0, (size_t)B * sizeof(int), st));
  for (int k0 = 0; k0 < N; k0 += kLuBlkNb) {
    const int nb = (N - k0 < kLuBlkNb) ? N - k0 : kLuBlkNb;
    // ---- panel: 16-column sub-panels of the outer block
    for (int j0 = k0; j0 < k0 + nb; j0 += kLuNb) {
      const int kb = (k0 + nb - j0 < kLuNb) ? k0 + nb - j0 : kLuNb;
      if ((rc = lu_launch_panel(K, piv, info, B, N, j0, kb, st))) return rc;
      if (nb > kb) {
        lu_swap_band_kernel<<<dim3(cdiv(nb, 128), B), 128, 0, st>>>(K, piv, N, j0, kb, k0, k0 + nb);
        IADMM_LAUNCH_CHECK("lu_swap_band_kernel");
      }
      const int band = k0 + nb - j0 - kb;                // block columns right of the sub-panel
      if (band > 0) {
        lu_trsm_nb_kernel<kLuNb><<<dim3(cdiv(band, kLuTrsmThreads), B), kLuTrsmThreads, kLuNb * kLuTrsmThreads * sizeof(float), st>>>(
            K, N, j0, kb, j0 + kb, k0 + nb);
        IADMM_LAUNCH_CHECK("lu_trsm_nb_kernel<16>");
        lu_update_band_kernel<<<dim3(cdiv(band, 128), cdiv(N - j0 - kb, 32), B), 128, 0, st>>>(K, N, j0, kb, k0 + nb);
        IADMM_LAUNCH_CHECK("lu_update_band_kernel");
      }
    }
    // ---- the block's interchanges on every other column, then U12 and the trailing update
    if (N > nb) {
      lu_swap_kernel<<<dim3(cdiv(N, 256), B), 256, 0, st>>>(K, piv, N, k0, nb);
      IADMM_LAUNCH_CHECK("lu_swap_kernel");
    }
    const int M = N - k0 - nb;
    if (M > 0) {
      lu_trsm_nb_kernel<kLuBlkNb><<<dim3(cdiv(M, kLuTrsmThreads), B), kLuTrsmThreads, kLuBlkNb * kLuTrsmThreads * sizeof(float), st>>>(
          K, N, k0, nb, k0 + nb, N);
      IADMM_LAUNCH_CHECK("lu_trsm_nb_kernel<128>");
      lu_split_l_kernel<<<dim3(cdiv(M, 256 / kLuBlkNb), B), 256, 0, st>>>(K, N, k0, nb, M, l_hi, l_lo);
      IADMM_LAUNCH_CHECK("lu_split_l_kernel");
      lu_split_ut_kernel<<<dim3(cdiv(M, 32), kLuBlkNb / 32, B), 256, 0, st>>>(K, N, k0, nb, M, u_hi, u_lo);
      IADMM_LAUNCH_CHECK("lu_split_ut_kernel");
      CUtensorMap m_lh, m_ll, m_uh, m_ul;
      if ((rc = lu_make_map(&m_lh, l_hi, B, N, M)) || (rc = lu_make_map(&m_ll, l_lo, B, N, M)) ||
          (rc = lu_make_map(&m_uh, u_hi, B, N, M)) || (rc = lu_make_map(&m_ul, u_lo, B, N, M)))
        return rc;
      LuGemmParams P;
      P.A = K; P.N = N; P.r0 = k0 + nb; P.M = M;
      P.tiles_m = cdiv(M, 2 * kTcBM); P.tiles_n = cdiv(M, kLgBN);
      P.units = (long)B * P.tiles_m * P.tiles_n;
      P.k_blocks = cdiv(nb, kLgBK);
      long pairs = num_sms / 2;
      if (P.units < pairs) pairs = P.units;
      lu_tf32_update_kernel<<<(unsigned)(2 * pairs), kLgThreads, kLgSmem, st>>>(m_lh, m_ll, m_uh, m_ul, P);
      IADMM_LAUNCH_CHECK("lu_tf32_update_kernel");
    }
  }
  lu_perm_kernel<<<B, 256, (size_t)N * sizeof(int), st>>>(piv, perm, N);
  IADMM_LAUNCH_CHECK("lu_perm_kernel");
  return IADMM_OK;
}

}  // extern "C"

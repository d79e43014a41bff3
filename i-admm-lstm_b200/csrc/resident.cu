// On-chip-resident variant of the K-step solve for SMALL instances: one persistent CTA per QP instance runs all K
// iterations without leaving the SM.
//
// Reference: the same loop as api.cu's streaming path -- models/lstm.py:47-96 per iteration, utils.py:68-71 for
// the residual traces, main.py:922-968 for the un-scaled residuals / objective / violations.
//
// Why: at n + m <= 256 and hidden_dim 64 (BASELINE config 1: n=100, 50+50, h=64) an iteration of the streaming
// path is six dependent launches of a few microseconds each -- launch latency, not bandwidth (profiles/README.md:
// 44 us per iteration under a CUDA graph).  Here everything an instance touches stays on its SM for the whole solve:
//   * Q and A0 (<= 80 KB fp32) are staged in shared memory once (or stay L2-resident when they do not fit);
//   * the hidden state H lives in shared memory directly in the tensor-core operand form (fp16 + e4m3 / fp16 hi/lo
//     images, 128-byte swizzled K-major rows) that the epilogue writes and the next iteration's MMAs read;
//   * the cell state C lives in registers (64 per thread), the gate weights U in shared memory (64 KB);
//   * the gate contraction is 2 x (M=128, N=256, K=64) tcgen05 MMAs into TMEM, issued at the START of the
//     iteration (it needs only H), so it overlaps the KKT mat-vecs that produce the gradient input;
//   * x, y, z, xv, the KKT temporaries and the residual reductions are shared-memory vectors.
// No grid-wide synchronisation, no global-memory traffic inside the loop except the trace rows.
// Instances are independent, so any batch size works (CTAs beyond the SM count simply queue).
#include "common.cuh"
#include "tc_ptx.cuh"
#include "gate_math.cuh"

#include <stdlib.h>

namespace iadmm {

constexpr int kResThreads = 512;                  // 16 warps: 4 per TMEM lane quarter, each owning 2 of a tile's 8 column chunks
constexpr int kResGroups = kResThreads / 128;     // column groups of the epilogue
constexpr int kResChunks = 8 / kResGroups;        // 8-unit chunks per thread and tile
constexpr int kResH = 64;                  // hidden units (one 64-wide K block, N = 256 gate columns)
constexpr int kResMaxN = 256;              // n + m: two 128-row accumulator tiles fill the 512 TMEM columns
constexpr int kResTileBytes = 128 * 128;   // one 128-row operand tile, 128-byte rows
constexpr int kResOperandBytes = 4 * 2 * kResTileBytes;   // A_hi | A_lo | B_hi | B_lo, 32 KB each
constexpr int kResSmemLimit = 227 * 1024;

struct ResArgs {
  const float *Q, *p, *A0, *zl, *zu, *sd, *se, *sc;
  float *x, *y, *z, *xv, *H, *C;
  float *pri, *dual, *pri_u, *dual_u, *metrics;   // trace bases (row 0), may be NULL
  const Sched* sched;                             // schedule row of the first iteration
  const float *wc, *bias, *wh, *bh, *scale;
  const void *uhi, *ulo;                          // [256][64] fp16 ; [256][64] fp16 (3 products) or [256][128] bytes (fp16+fp8)
  int B, n, m, num_ineq, K, flags;
  float sigma;
  int cache_mats;                                 // Q and A0 staged in shared memory
};

// byte offset of 16-byte chunk `j` of row `r` inside a 128-byte-swizzled K-major operand tile
__device__ __forceinline__ uint32_t sw128_off(int r, int j) { return (uint32_t)((r >> 3) * 1024 + (r & 7) * 128 + ((j ^ (r & 7)) << 4)); }

template <int NPROD>
__device__ __forceinline__ void store_hidden8(uint8_t* a_hi, uint8_t* a_lo, int row, int unit0, const float (&hnew)[8]) {
  uint32_t hi[4], lo[4], res[2], crs[2];
  split_hidden8<NPROD>(hnew, hi, lo, res, crs);
  const int t = row >> 7, r = row & 127;
  uint8_t* th = a_hi + t * kResTileBytes;
  uint8_t* tl = a_lo + t * kResTileBytes;
  *reinterpret_cast<uint4*>(th + sw128_off(r, unit0 >> 3)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
  if (NPROD == 3) *reinterpret_cast<uint4*>(tl + sw128_off(r, unit0 >> 3)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  if (NPROD == 2) {      // bytes [0,64) of the row: e4m3 residual; [64,128): e4m3 coarse copy
    const int within = unit0 & 15;
    *reinterpret_cast<uint2*>(tl + sw128_off(r, unit0 >> 4) + within)       = make_uint2(res[0], res[1]);
    *reinterpret_cast<uint2*>(tl + sw128_off(r, 4 + (unit0 >> 4)) + within) = make_uint2(crs[0], crs[1]);
  }
}

struct ResSmem {
  uint8_t *a_hi, *a_lo, *b_hi, *b_lo;
  float *w0, *w1, *bias, *wh;                       // gate-column parameters (interleaved 4*unit + gate)
  float *x, *y, *z, *xt, *v, *p, *zl, *zu;          // iterates (xv = [xt; v]) and instance vectors
  float *w1v, *w2v, *g, *t0, *t1, *qx, *ax, *aty;   // KKT temporaries (w = [w1v; w2v])
  float *xo, *yo, *zo;                              // the iterate before the last tail update (linear-system residual)
  float *cp;                                        // [parts][2][cw] column partials (KKT phases)
  float *head;                                      // [groups][256] head partials (cell phase; aliases cp)
  uint64_t* bar;
  uint32_t* tmem_slot;
  float* mat;                                       // stacked [Q; A0], (n+m) rows of `ld` floats, when cached
};

__host__ __device__ inline int r4(int v) { return (v + 3) & ~3; }
// leading dimension of the cached matrix: odd, so that one-row-per-thread dot products are bank-conflict free
__host__ __device__ inline int res_ld(int n) { return n | 1; }
__host__ __device__ inline size_t res_vec_floats(int n, int m) {
  const int N = n + m;
  // x y z xt v p zl zu | w1v w2v g t0 t1 qx ax aty | xo yo zo   (each rounded up to a multiple of 4 floats)
  return (size_t)r4(n) + r4(m) + r4(m) + r4(n) + r4(m) + r4(n) + r4(m) + r4(m) + r4(n) + r4(m) + r4(N) + r4(N) + r4(N) + r4(n) +
         r4(m) + r4(n) + r4(n) + r4(m) + r4(m);
}
__host__ __device__ inline size_t res_fixed_bytes(int n, int m) {
  return 1024 /*alignment slack*/ + kResOperandBytes + (3 * 256 + 64) * sizeof(float) + res_vec_floats(n, m) * sizeof(float) +
         2 * kResThreads * sizeof(float) + 64;
}

// `base` is the 1024-byte aligned start of the dynamic shared memory (pointer arithmetic only, so that the compiler
// keeps the shared address space and emits LDS/STS)
__device__ __forceinline__ void res_carve(uint8_t* base, int n, int m, ResSmem& S) {
  S.a_hi = base; S.a_lo = base + 2 * kResTileBytes; S.b_hi = base + 4 * kResTileBytes; S.b_lo = base + 6 * kResTileBytes;
  double* dp = reinterpret_cast<double*>(base + kResOperandBytes);
  S.bar = reinterpret_cast<uint64_t*>(dp); dp += 2;
  S.tmem_slot = reinterpret_cast<uint32_t*>(dp); dp += 2;
  float* fp = reinterpret_cast<float*>(dp);
  const int N = n + m;
  S.w0 = fp; fp += 256; S.w1 = fp; fp += 256; S.bias = fp; fp += 256; S.wh = fp; fp += 64;
  S.cp = fp; S.head = fp; fp += 2 * kResThreads;
  S.x = fp; fp += r4(n); S.y = fp; fp += r4(m); S.z = fp; fp += r4(m); S.xt = fp; fp += r4(n); S.v = fp; fp += r4(m);
  S.p = fp; fp += r4(n); S.zl = fp; fp += r4(m); S.zu = fp; fp += r4(m);
  S.w1v = fp; fp += r4(n); S.w2v = fp; fp += r4(m); S.g = fp; fp += r4(N); S.t0 = fp; fp += r4(N); S.t1 = fp; fp += r4(N);
  S.qx = fp; fp += r4(n); S.ax = fp; fp += r4(m); S.aty = fp; fp += r4(n);
  S.xo = fp; fp += r4(n); S.yo = fp; fp += r4(m); S.zo = fp; fp += r4(m);
  S.mat = fp;
}

// ---- KKT mat-vecs ----------------------------------------------------------------------------------------------------
// (a) matrix cached in shared memory with an odd leading dimension: ONE THREAD PER ROW for row dots (the lanes of a
//     warp read addresses `ld` apart: conflict free; the vector is a broadcast float4), one thread per column (and
//     row group) for column sums.
template <bool TWO>
__device__ __forceinline__ void res_row_dot_thread(const float* row, int n, const float* u0, const float* u1, float& d0, float& d1) {
  float a0 = 0.f, a1 = 0.f;
  int c = 0;
  for (; c + 4 <= n; c += 4) {
    const float m0 = row[c], m1 = row[c + 1], m2 = row[c + 2], m3 = row[c + 3];
    const float4 p = *reinterpret_cast<const float4*>(u0 + c);
    a0 = fmaf(m0, p.x, a0); a0 = fmaf(m1, p.y, a0); a0 = fmaf(m2, p.z, a0); a0 = fmaf(m3, p.w, a0);
    if (TWO) {
      const float4 q = *reinterpret_cast<const float4*>(u1 + c);
      a1 = fmaf(m0, q.x, a1); a1 = fmaf(m1, q.y, a1); a1 = fmaf(m2, q.z, a1); a1 = fmaf(m3, q.w, a1);
    }
  }
  for (; c < n; ++c) {
    const float mm = row[c];
    a0 = fmaf(mm, u0[c], a0);
    if (TWO) a1 = fmaf(mm, u1[c], a1);
  }
  d0 = a0; d1 = a1;
}
// column sums over rows [0, rows) of a matrix block: thread (part, c) takes a contiguous group of rows (multiple of 4,
// so the vector entries are broadcast float4 reads)
template <bool TWO>
__device__ __forceinline__ void res_col_sum_thread(const float* Mc, int ld, int rows, int part, int parts, const float* u0,
                                                   const float* u1, float& s0, float& s1) {
  float a0 = 0.f, a1 = 0.f;
  const int per = r4((rows + parts - 1) / parts);
  int r = part * per;
  const int r_end = min(rows, r + per);
  const float* pm = Mc + (size_t)r * ld;
  for (; r + 4 <= r_end; r += 4, pm += 4 * ld) {
    const float m0 = pm[0], m1 = pm[ld], m2 = pm[2 * ld], m3 = pm[3 * ld];
    const float4 p = *reinterpret_cast<const float4*>(u0 + r);
    a0 = fmaf(m0, p.x, a0); a0 = fmaf(m1, p.y, a0); a0 = fmaf(m2, p.z, a0); a0 = fmaf(m3, p.w, a0);
    if (TWO) {
      const float4 q = *reinterpret_cast<const float4*>(u1 + r);
      a1 = fmaf(m0, q.x, a1); a1 = fmaf(m1, q.y, a1); a1 = fmaf(m2, q.z, a1); a1 = fmaf(m3, q.w, a1);
    }
  }
  for (; r < r_end; ++r, pm += ld) {
    const float a = pm[0];
    a0 = fmaf(a, u0[r], a0);
    if (TWO) a1 = fmaf(a, u1[r], a1);
  }
  s0 = a0; s1 = a1;
}
// (b) matrix in global memory (L2 resident): one WARP per row so the reads coalesce
__device__ __forceinline__ void res_row_dots_warp(const float* __restrict__ M, int n, int rows, const float* u0, const float* u1,
                                                  float* out0, float* out1, int warp, int lane) {
  for (int r = warp; r < rows; r += kResThreads / 32) {
    const float* row = M + (size_t)r * n;
    float d0 = 0.f, d1 = 0.f;
    for (int c = lane; c < n; c += 32) {
      const float a = __ldg(row + c);
      d0 = fmaf(a, u0[c], d0);
      if (u1) d1 = fmaf(a, u1[c], d1);
    }
    d0 = warp_sum(d0);
    if (u1) d1 = warp_sum(d1);
    if (lane == 0) { out0[r] = d0; if (u1) out1[r] = d1; }
  }
}
__device__ __forceinline__ float res_col_total(const float* cp, int cw, int which, int c) {
  float s = 0.f;
  for (int part = 0; part < kResThreads / cw; ++part) s += cp[(part * 2 + which) * cw + c];
  return s;
}

// residual norms / metrics of the iterate (x, y, z) from qx = Q x, ax = A0 x, aty = A0^T y (all in shared memory);
// same quantities, accumulation type (double) and output layout as kkt_combine1_kernel.  Five warps take one
// quantity group each and write their trace entries themselves: no block-wide reduction, no barrier.
__device__ __forceinline__ double warp_sum_double(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
  return v;
}
__device__ __forceinline__ void res_trace_row(const ResArgs& A, const ResSmem& S, int b, int row, int warp, int lane) {
  if (warp > 5) return;
  const int n = A.n, m = A.m;
  const bool want_met = A.metrics != nullptr;
  const bool unscaled = (A.sd != nullptr) && (A.pri_u || A.dual_u || want_met);
  const float cscale = unscaled ? A.sc[b] : 1.f;
  const size_t B = A.B, o = (size_t)row * B + b;
  float* mt = want_met ? A.metrics + (size_t)row * kMetricRows * B : nullptr;
  if (warp == 0) {                                   // dual residual || Q x + p + A0^T y ||
    double s = 0.0, su = 0.0;
    for (int j = lane; j < n; j += 32) {
      const float r = __fadd_rn(__fadd_rn(S.qx[j], S.p[j]), S.aty[j]);
      s += (double)r * (double)r;
      if (unscaled) { const float ru = r / (cscale * A.sd[(size_t)b * n + j]); su += (double)ru * (double)ru; }
    }
    s = warp_sum_double(s);
    if (unscaled) su = warp_sum_double(su);
    if (lane == 0) {
      if (A.dual) A.dual[o] = (float)sqrt(s);
      if (unscaled && A.dual_u) A.dual_u[o] = (float)sqrt(su);
    }
  } else if (warp == 1) {                            // primal residual || A0 x - z ||
    double s = 0.0, su = 0.0;
    for (int i = lane; i < m; i += 32) {
      const float r = __fsub_rn(S.ax[i], S.z[i]);
      s += (double)r * (double)r;
      if (unscaled) { const float ru = r / A.se[(size_t)b * m + i]; su += (double)ru * (double)ru; }
    }
    s = warp_sum_double(s);
    if (unscaled) su = warp_sum_double(su);
    if (lane == 0) {
      if (A.pri) A.pri[o] = (float)sqrt(s);
      if (unscaled && A.pri_u) A.pri_u[o] = (float)sqrt(su);
    }
  } else if (!want_met) {
    return;
  } else if (warp == 5) {                            // || K xv - rhs || (main.py:952); elements staged in S.g by the caller
    double s = 0.0;
    for (int i = lane; i < n + m; i += 32) s += (double)S.g[i] * (double)S.g[i];
    s = warp_sum_double(s);
    if (lane == 0) mt[5 * B + b] = (float)sqrt(s);
  } else if (warp == 2) {                            // objective 0.5 x^T Q x + p^T x (main.py:950)
    double s = 0.0;
    for (int j = lane; j < n; j += 32) s += (double)S.x[j] * (0.5 * (double)S.qx[j] + (double)S.p[j]);
    s = warp_sum_double(s);
    if (lane == 0) mt[0 * B + b] = (float)(unscaled ? s / (double)cscale : s);
  } else {                                           // warp 3: inequality rows, warp 4: equality rows (main.py:957-968)
    const bool ineq = (warp == 3);
    const int i0 = ineq ? 0 : A.num_ineq, i1 = ineq ? A.num_ineq : m;
    double s = 0.0; float mx = 0.f;
    for (int i = i0 + lane; i < i1; i += 32) {
      const float einv = unscaled ? 1.0f / A.se[(size_t)b * m + i] : 1.0f;
      const float dv = (S.ax[i] - S.zu[i]) * einv;
      const float q = ineq ? fmaxf(dv, 0.f) : fabsf(dv);
      mx = fmaxf(mx, q); s += (double)q;
    }
    s = warp_sum_double(s); mx = warp_max(mx);
    if (lane == 0) {
      const int cnt = i1 - i0;
      mt[(ineq ? 1 : 3) * B + b] = mx;
      mt[(ineq ? 2 : 4) * B + b] = cnt > 0 ? (float)(s / cnt) : 0.f;
    }
  }
}

template <int NPROD, bool CACHED>
__global__ void __launch_bounds__(kResThreads, 1) solve_resident_kernel(const ResArgs A) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  ResSmem S;
  const int n = A.n, m = A.m, N = n + m;
  res_carve(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u), n, m, S);
  const int b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int quarter = warp & 3, grp = warp >> 2;
  const int ntiles = (N + 127) >> 7;
  const bool want_trace = A.pri || A.dual || A.pri_u || A.dual_u || A.metrics;
  const int ld = res_ld(n);

  // ---------------- one-time staging ----------------
  for (int i = tid; i < 256; i += kResThreads) {
    S.w0[i] = A.wc[i]; S.w1[i] = A.wc[256 + i]; S.bias[i] = A.bias[i];
    if (i < kResH) S.wh[i] = A.wh[i];
  }
  {
    uint4* za = reinterpret_cast<uint4*>(S.a_hi);                    // A_hi | A_lo: zero (rows >= N stay zero forever)
    for (int i = tid; i < 4 * kResTileBytes / 16; i += kResThreads) za[i] = make_uint4(0, 0, 0, 0);
    const uint4* uh = reinterpret_cast<const uint4*>(A.uhi);
    const uint4* ul = reinterpret_cast<const uint4*>(A.ulo);
    for (int i = tid; i < 256 * 8; i += kResThreads) {
      const int r = i >> 3, j = i & 7;
      *reinterpret_cast<uint4*>(S.b_hi + sw128_off(r, j)) = __ldg(uh + i);
      if (NPROD != 1) *reinterpret_cast<uint4*>(S.b_lo + sw128_off(r, j)) = __ldg(ul + i);
    }
  }
  for (int i = tid; i < r4(n); i += kResThreads) {                   // padding lanes of the float4 reads: zero
    const bool ok = i < n;
    S.x[i] = ok ? A.x[(size_t)b * n + i] : 0.f; S.p[i] = ok ? A.p[(size_t)b * n + i] : 0.f;
    S.xt[i] = ok ? A.xv[(size_t)b * N + i] : 0.f; S.w1v[i] = 0.f;
  }
  for (int i = tid; i < r4(m); i += kResThreads) {
    const bool ok = i < m;
    S.y[i] = ok ? A.y[(size_t)b * m + i] : 0.f; S.z[i] = ok ? A.z[(size_t)b * m + i] : 0.f;
    S.zl[i] = ok ? A.zl[(size_t)b * m + i] : 0.f; S.zu[i] = ok ? A.zu[(size_t)b * m + i] : 0.f;
    S.v[i] = ok ? A.xv[(size_t)b * N + n + i] : 0.f; S.w2v[i] = 0.f;
  }
  const float* Qg = A.Q + (size_t)b * n * n;
  const float* Ag = (m > 0) ? A.A0 + (size_t)b * m * n : nullptr;
  if (CACHED) {
    for (int i = tid; i < n * n; i += kResThreads) S.mat[(i / n) * ld + (i % n)] = __ldg(Qg + i);
    for (int i = tid; i < m * n; i += kResThreads) S.mat[(n + i / n) * ld + (i % n)] = __ldg(Ag + i);
  }
  const float* Ms = S.mat;                                           // cached: stacked [Q; A0], leading dimension ld
  const float* Msa = S.mat + (size_t)n * ld;

  if (tid == 0) {
    mbar_init(smem_u32(S.bar), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(S.tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  __syncthreads();          // zero-filled A tiles visible before the state is written into them

  // ---------------- state: C into registers, H into the operand tiles ----------------
  float creg[2][kResChunks][8];
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    const int row = t * 128 + quarter * 32 + lane;
#pragma unroll
    for (int cc = 0; cc < kResChunks; ++cc) {
      const int unit0 = (grp * kResChunks + cc) * 8;
      if (row < N) {
        const size_t o = ((size_t)b * N + row) * kResH + unit0;
        ld_global_v8(A.C + o, creg[t][cc]);
        if (!(A.flags & IADMM_F_ZERO_STATE)) {
          float hv[8];
          ld_global_v8(A.H + o, hv);
          store_hidden8<NPROD>(S.a_hi, S.a_lo, row, unit0, hv);
        }
      } else {
#pragma unroll
        for (int u = 0; u < 8; ++u) creg[t][cc][u] = 0.f;
      }
    }
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");       // operand tiles were written by the generic proxy
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *S.tmem_slot;
  const float dequant = A.scale[1];
  const float b_h = A.bh[0];
  const uint32_t idesc = make_idesc_f16(256);
  const int cw = (n <= 32) ? 32 : (n <= 64) ? 64 : (n <= 128) ? 128 : 256;      // column-sum group width
  const int parts = kResThreads / cw, part = tid / cw, col = tid % cw;

  for (int k = 0; k < A.K; ++k) {
    const Sched sk = A.sched[k];
    // ---- gate contraction H @ U: needs only H, so it is issued first and runs under the KKT phase ----
    if (tid == 0) {
      for (int t = 0; t < ntiles; ++t) {
        const uint32_t d_tmem = tmem_base + (uint32_t)(t * 256);
        const uint32_t ah = smem_u32(S.a_hi) + t * kResTileBytes, al = smem_u32(S.a_lo) + t * kResTileBytes;
        const uint32_t bh = smem_u32(S.b_hi), bl = smem_u32(S.b_lo);
        uint32_t acc = 0;
#pragma unroll
        for (int ks = 0; ks < kResH / kTcUK; ++ks) {
          const uint32_t koff = (uint32_t)(ks * kTcUK * 2);
          if (NPROD == 3) {
            tc_mma_f16(d_tmem, make_smem_desc_sw128(al + koff), make_smem_desc_sw128(bh + koff), idesc, acc); acc = 1;
            tc_mma_f16(d_tmem, make_smem_desc_sw128(ah + koff), make_smem_desc_sw128(bl + koff), idesc, 1);
          } else if (NPROD == 2 && (ks & 1) == 0) {
            const uint32_t koff8 = (uint32_t)(ks * kTcUK);
            tc_mma_f8(d_tmem, make_smem_desc_sw128(al + koff8), make_smem_desc_sw128(bl + 64 + koff8), idesc, acc); acc = 1;   // (H - fp16 H) U
            tc_mma_f8(d_tmem, make_smem_desc_sw128(al + 64 + koff8), make_smem_desc_sw128(bl + koff8), idesc, 1);              // H (U - fp16 U)
          }
          tc_mma_f16(d_tmem, make_smem_desc_sw128(ah + koff), make_smem_desc_sw128(bh + koff), idesc, acc); acc = 1;
        }
      }
      tc_commit(smem_u32(S.bar));
    }

    // ---- KKT pass 1: [Q; A0] {x~, x} (row dots) and A0^T {v, y} (column sums) ----
    if (CACHED) {
      if (tid < N) res_row_dot_thread<true>(Ms + (size_t)tid * ld, n, S.xt, S.x, S.t0[tid], S.t1[tid]);
      if (m > 0) {
        float s0, s1;
        res_col_sum_thread<true>(Msa + col, ld, (col < n) ? m : 0, part, parts, S.v, S.y, s0, s1);
        S.cp[(part * 2 + 0) * cw + col] = s0; S.cp[(part * 2 + 1) * cw + col] = s1;
      }
    } else {
      res_row_dots_warp(Qg, n, n, S.xt, S.x, S.t0, S.t1, warp, lane);
      if (m > 0) {
        res_row_dots_warp(Ag, n, m, S.xt, S.x, S.t0 + n, S.t1 + n, warp, lane);
        float s0, s1;
        res_col_sum_thread<true>(Ag + col, n, (col < n) ? m : 0, part, parts, S.v, S.y, s0, s1);
        S.cp[(part * 2 + 0) * cw + col] = s0; S.cp[(part * 2 + 1) * cw + col] = s1;
      }
    }
    __syncthreads();
    if (tid < n) {
      const float atv = (m > 0) ? res_col_total(S.cp, cw, 0, tid) : 0.f;
      const float aty = (m > 0) ? res_col_total(S.cp, cw, 1, tid) : 0.f;
      const float kxv = __fadd_rn(__fadd_rn(S.t0[tid], __fmul_rn(A.sigma, S.xt[tid])), atv);
      const float rhs = __fsub_rn(__fmul_rn(A.sigma, S.x[tid]), S.p[tid]);
      S.w1v[tid] = __fsub_rn(kxv, rhs);
      S.qx[tid] = S.t1[tid];
      S.aty[tid] = aty;
      if (k > 0 && A.metrics) S.g[tid] = __fsub_rn(kxv, __fsub_rn(__fmul_rn(A.sigma, S.xo[tid]), S.p[tid]));
    } else if (tid < N) {
      const int i = tid - n;
      const float inv = (i < A.num_ineq) ? sk.inv_rho_ineq : sk.inv_rho_eq;
      const float kxv = __fsub_rn(S.t0[tid], __fmul_rn(inv, S.v[i]));
      const float rhs = __fsub_rn(S.z[i], __fmul_rn(inv, S.y[i]));
      S.w2v[i] = __fsub_rn(kxv, rhs);
      S.ax[i] = S.t1[tid];
      if (k > 0 && A.metrics) {                      // previous iteration's penalties and pre-update iterate
        const float pinv = (i < A.num_ineq) ? A.sched[k - 1].inv_rho_ineq : A.sched[k - 1].inv_rho_eq;
        S.g[tid] = __fsub_rn(__fsub_rn(S.t0[tid], __fmul_rn(pinv, S.v[i])), __fsub_rn(S.zo[i], __fmul_rn(pinv, S.yo[i])));
      }
    }
    __syncthreads();
    if (k > 0 && want_trace) res_trace_row(A, S, b, k - 1, warp, lane);   // residuals of the iterate entering this iteration

    // ---- KKT pass 2: g = K^T w: Q^T w1 and A0^T w2 (column sums), A0 w1 (row dots) ----
    {
      float sq, sa = 0.f, dummy;
      if (CACHED) {
        res_col_sum_thread<false>(Ms + col, ld, (col < n) ? n : 0, part, parts, S.w1v, nullptr, sq, dummy);
        if (m > 0) res_col_sum_thread<false>(Msa + col, ld, (col < n) ? m : 0, part, parts, S.w2v, nullptr, sa, dummy);
        if (tid >= n && tid < N) res_row_dot_thread<false>(Ms + (size_t)tid * ld, n, S.w1v, nullptr, S.t0[tid], dummy);
      } else {
        res_col_sum_thread<false>(Qg + col, n, (col < n) ? n : 0, part, parts, S.w1v, nullptr, sq, dummy);
        if (m > 0) {
          res_col_sum_thread<false>(Ag + col, n, (col < n) ? m : 0, part, parts, S.w2v, nullptr, sa, dummy);
          res_row_dots_warp(Ag, n, m, S.w1v, nullptr, S.t0 + n, nullptr, warp, lane);
        }
      }
      S.cp[(part * 2 + 0) * cw + col] = sq; S.cp[(part * 2 + 1) * cw + col] = sa;
    }
    __syncthreads();
    if (tid < n) {
      const float qtw = res_col_total(S.cp, cw, 0, tid);
      const float atw = (m > 0) ? res_col_total(S.cp, cw, 1, tid) : 0.f;
      S.g[tid] = __fadd_rn(__fadd_rn(qtw, __fmul_rn(A.sigma, S.w1v[tid])), atw);
    } else if (tid < N) {
      const int i = tid - n;
      const float inv = (i < A.num_ineq) ? sk.inv_rho_ineq : sk.inv_rho_eq;
      S.g[tid] = __fsub_rn(S.t0[tid], __fmul_rn(inv, S.w2v[i]));
    }
    __syncthreads();

    // ---- LSTM cell on the accumulators (models/lstm.py:74-80) ----
    mbar_wait(smem_u32(S.bar), (uint32_t)(k & 1));
    tc_fence_after();
    const bool last = (k == A.K - 1);
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      const int row = t * 128 + quarter * 32 + lane;
      if (t * 128 + quarter * 32 < N) {                              // warp-uniform: this warp owns live rows of tile t
        const bool row_ok = row < N;
        const float xr = row_ok ? (row < n ? S.xt[row] : S.v[row - n]) : 0.f, gr = row_ok ? S.g[row] : 0.f;
        float hp = 0.f;
        const u64 xr2 = bc2(xr), gr2 = bc2(gr), dq2 = bc2(dequant);
#pragma unroll
        for (int cc = 0; cc < kResChunks; ++cc) {
          const int chunk = grp * kResChunks + cc;
          const int unit0 = chunk * 8;
          uint32_t acc[32];
          tc_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(t * 256 + chunk * 32), acc);
          tc_wait_ld();
          if (row_ok) {
            float hnew[8];
            const float4* w0 = reinterpret_cast<const float4*>(S.w0 + chunk * 32);
            const float4* w1 = reinterpret_cast<const float4*>(S.w1 + chunk * 32);
            const float4* bb = reinterpret_cast<const float4*>(S.bias + chunk * 32);
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              const float4 a0 = w0[u], a1 = w1[u], ab = bb[u];
              // pre-activations of the gate pairs (i,f) and (o,u) two-wide (FFMA2): lane by lane the scalar fmaf chain
              const u64 pif = fma2(pk2(__uint_as_float(acc[u * 4 + 0]), __uint_as_float(acc[u * 4 + 1])), dq2,
                                   fma2(gr2, pk2(a1.x, a1.y), fma2(xr2, pk2(a0.x, a0.y), pk2(ab.x, ab.y))));
              const u64 pou = fma2(pk2(__uint_as_float(acc[u * 4 + 2]), __uint_as_float(acc[u * 4 + 3])), dq2,
                                   fma2(gr2, pk2(a1.z, a1.w), fma2(xr2, pk2(a0.z, a0.w), pk2(ab.z, ab.w))));
              float gi, gf, go, gu;
              gates4_shared_rcp_x2(pif, pou, gi, gf, go, gu);
              const float cn = __fadd_rn(__fmul_rn(gi, gu), __fmul_rn(gf, creg[t][cc][u]));
              const float hn = __fmul_rn(go, tanh_exp(cn));
              creg[t][cc][u] = cn;
              hnew[u] = hn;
              hp = fmaf(hn, S.wh[unit0 + u], hp);
            }
            store_hidden8<NPROD>(S.a_hi, S.a_lo, row, unit0, hnew);
            if (last) st_global_v8(A.H + ((size_t)b * N + row) * kResH + unit0, hnew);
          }
        }
        if (row_ok) S.head[grp * 256 + row] = hp;
      }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // new H images -> visible to the next MMAs
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    // ---- tail (models/lstm.py:80-94), every product and sum rounded as the reference rounds it ----
    if (tid < N) {
      float head = 0.f;
#pragma unroll
      for (int q = 0; q < kResGroups; ++q) head += S.head[q * 256 + tid];
      head = __fadd_rn(head, b_h);
      if (tid < n) {
        const float xvn = __fsub_rn(S.xt[tid], head);
        S.xt[tid] = xvn;
        const float xold = S.x[tid];
        S.xo[tid] = xold;
        S.x[tid] = __fadd_rn(__fmul_rn(sk.alpha, xvn), __fmul_rn(sk.one_minus_alpha, xold));
      } else {
        const int i = tid - n;
        const float xvn = __fsub_rn(S.v[i], head);
        S.v[i] = xvn;
        const bool eq = i >= A.num_ineq;
        const float rho = eq ? sk.rho_eq : sk.rho_ineq, inv = eq ? sk.inv_rho_eq : sk.inv_rho_ineq;
        const float yo = S.y[i], zo = S.z[i];
        S.yo[i] = yo; S.zo[i] = zo;
        const float zmid = __fadd_rn(zo, __fmul_rn(inv, __fsub_rn(xvn, yo)));
        const float zc = fmaxf(fminf(__fadd_rn(zmid, __fmul_rn(inv, yo)), S.zu[i]), S.zl[i]);
        S.z[i] = zc;
        S.y[i] = __fadd_rn(yo, __fmul_rn(rho, __fsub_rn(zmid, zc)));
      }
    }
    __syncthreads();
  }

  // ---------------- trailing residual row, state write-back ----------------
  if (want_trace && A.K > 0 && !(A.flags & IADMM_F_SKIP_FINAL_RESID)) {
    if (CACHED) {
      if (tid < N) res_row_dot_thread<true>(Ms + (size_t)tid * ld, n, S.xt, S.x, S.t0[tid], S.t1[tid]);
      if (m > 0) {
        float s0, s1;
        res_col_sum_thread<true>(Msa + col, ld, (col < n) ? m : 0, part, parts, S.v, S.y, s0, s1);
        S.cp[(part * 2 + 0) * cw + col] = s0; S.cp[(part * 2 + 1) * cw + col] = s1;
      }
    } else {
      res_row_dots_warp(Qg, n, n, S.xt, S.x, S.t0, S.t1, warp, lane);
      if (m > 0) {
        res_row_dots_warp(Ag, n, m, S.xt, S.x, S.t0 + n, S.t1 + n, warp, lane);
        float s0, s1;
        res_col_sum_thread<true>(Ag + col, n, (col < n) ? m : 0, part, parts, S.v, S.y, s0, s1);
        S.cp[(part * 2 + 0) * cw + col] = s0; S.cp[(part * 2 + 1) * cw + col] = s1;
      }
    }
    __syncthreads();
    const Sched sl = A.sched[A.K - 1];
    if (tid < n) {
      const float atv = (m > 0) ? res_col_total(S.cp, cw, 0, tid) : 0.f;
      S.qx[tid] = S.t1[tid]; S.aty[tid] = (m > 0) ? res_col_total(S.cp, cw, 1, tid) : 0.f;
      const float kxv = __fadd_rn(__fadd_rn(S.t0[tid], __fmul_rn(A.sigma, S.xt[tid])), atv);
      S.g[tid] = __fsub_rn(kxv, __fsub_rn(__fmul_rn(A.sigma, S.xo[tid]), S.p[tid]));
    } else if (tid < N) {
      const int i = tid - n;
      S.ax[i] = S.t1[tid];
      const float pinv = (i < A.num_ineq) ? sl.inv_rho_ineq : sl.inv_rho_eq;
      S.g[tid] = __fsub_rn(__fsub_rn(S.t0[tid], __fmul_rn(pinv, S.v[i])), __fsub_rn(S.zo[i], __fmul_rn(pinv, S.yo[i])));
    }
    __syncthreads();
    res_trace_row(A, S, b, A.K - 1, warp, lane);
  }
  for (int i = tid; i < n; i += kResThreads) { A.x[(size_t)b * n + i] = S.x[i]; A.xv[(size_t)b * N + i] = S.xt[i]; }
  for (int i = tid; i < m; i += kResThreads) {
    A.y[(size_t)b * m + i] = S.y[i]; A.z[(size_t)b * m + i] = S.z[i]; A.xv[(size_t)b * N + n + i] = S.v[i];
  }
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    const int row = t * 128 + quarter * 32 + lane;
    if (row < N) {
#pragma unroll
      for (int cc = 0; cc < kResChunks; ++cc)
        st_global_v8(A.C + ((size_t)b * N + row) * kResH + (grp * kResChunks + cc) * 8, creg[t][cc]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
bool resident_eligible(int n, int m, int h, int nprod) {
  if (h != kResH || n + m > kResMaxN || nprod < 1 || nprod > 3) return false;
  return res_fixed_bytes(n, m) <= (size_t)kResSmemLimit;
}

int launch_solve_resident(const void* packed, const WeightLayout& L, const float* Q, const float* p, const float* A0,
                          const float* zl, const float* zu, const float* sd, const float* se, const float* sc, float* x, float* y,
                          float* z, float* xv, float* H, float* C, float* pri, float* dual, float* pri_u, float* dual_u,
                          float* metrics, int B, int n, int m, int num_ineq, int t0, int K, float sigma, int nprod, int flags,
                          cudaStream_t st) {
  const char* base = static_cast<const char*>(packed);
  ResArgs A;
  A.Q = Q; A.p = p; A.A0 = A0; A.zl = zl; A.zu = zu; A.sd = sd; A.se = se; A.sc = sc;
  A.x = x; A.y = y; A.z = z; A.xv = xv; A.H = H; A.C = C;
  A.pri = pri; A.dual = dual; A.pri_u = pri_u; A.dual_u = dual_u;
  A.metrics = (metrics && (zu || m == 0)) ? metrics : nullptr;
  A.sched = reinterpret_cast<const Sched*>(base + L.off_sched) + t0;
  A.wc = reinterpret_cast<const float*>(base + L.off_wc);
  A.bias = reinterpret_cast<const float*>(base + L.off_bias);
  A.wh = reinterpret_cast<const float*>(base + L.off_wh);
  A.bh = reinterpret_cast<const float*>(base + L.off_bh);
  A.scale = reinterpret_cast<const float*>(base + L.off_scale);
  A.uhi = base + L.off_uhi;
  A.ulo = (nprod == 2) ? base + L.off_uq8 : base + L.off_ulo;
  A.B = B; A.n = n; A.m = m; A.num_ineq = num_ineq; A.K = K; A.flags = flags; A.sigma = sigma;
  const size_t fixed = res_fixed_bytes(n, m);
  const size_t mats = (size_t)(n + m) * res_ld(n) * sizeof(float);
  A.cache_mats = (fixed + mats <= (size_t)kResSmemLimit) ? 1 : 0;
  const size_t smem = fixed + (A.cache_mats ? mats : 0);
  static PerDeviceOnce attr[8];
  auto go = [&](auto kernel) -> int {
    const int slot = nprod * 2 + A.cache_mats - 2;
    int rc2;
    if ((rc2 = ensure_dyn_smem(kernel, kResSmemLimit, &attr[slot]))) return rc2;
    kernel<<<B, kResThreads, smem, st>>>(A);
    return IADMM_OK;
  };
  int rc;
  if (A.cache_mats) rc = (nprod == 3) ? go(solve_resident_kernel<3, true>) : (nprod == 2) ? go(solve_resident_kernel<2, true>) : go(solve_resident_kernel<1, true>);
  else              rc = (nprod == 3) ? go(solve_resident_kernel<3, false>) : (nprod == 2) ? go(solve_resident_kernel<2, false>) : go(solve_resident_kernel<1, false>);
  if (rc) return rc;
  IADMM_LAUNCH_CHECK("solve_resident_kernel");
  return IADMM_OK;
}

}  // namespace iadmm

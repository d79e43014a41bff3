// Training path: one differentiable I-ADMM-LSTM iteration (forward that saves activations + hand-written
// backward) and the backward of primal_dual_loss.
//
// Reference: the autograd tape PyTorch builds through models/lstm.py:47-96 and utils.py:68-71 inside the
// truncated-BPTT loop main.py:336-358.  Here the backward of one iteration is derived by hand
// (notation: a bar is an adjoint, ' marks the iteration's outputs):
//   tail     y' = y + rho (z~ - z'),  z' = clip(z~ + y/rho),  x' = alpha x~' + (1-alpha) x,  z~ = z + (v' - y)/rho
//   step     xv' = xv - (H' W_h + b_h)
//   cell     H' = O tanh(C'), C' = I U~ + F C, gates = act([xv, g] W + H U + b)
//   KKT      g = K^T w,  w = K xv - rhs(x, y, z)      (K symmetric in structure: the adjoint passes ARE the
//            forward passes: w_bar = K g_bar, xv_bar += K^T w_bar, rhs_bar = -w_bar)
// so the two streaming KKT kernels of the forward are reused unchanged, and the only new heavy work is
// two plain fp32 GEMMs (H_bar = D U^T, U_bar = H^T D) plus column sums for the small parameters.
// This is the fp32 CUDA-core path (correctness first: gradients match torch.autograd through the float64 restatement of the reference
// to ~1e-5); tensor-core backward kernels are future work (DESIGN.md section 7).
#include "common.cuh"

#include <stdlib.h>

namespace iadmm {

int launch_kkt_pass1_plain(const KktDims& d, const float* Q, const float* A0, const float* x, const float* y,
                           const KktScratch& s, cudaStream_t st);
// gemm_tc.cu
int launch_tc_gemm_nt(const __half* A_hi, const __half* A_lo, const __half* B_hi, const __half* B_lo, float* C,
                      const float* scale, long M, long N, long K, long lda, long ldb, long ldc, cudaStream_t st,
                      int splits = 1, float* part = nullptr, int prod_mask = 7);
int tc_gemm_pick_splits(long M, long N, long K, int num_sms, int max_splits);
constexpr int kMaxSplitK = 16;
int launch_absmax(const float* X, size_t count, float* out, cudaStream_t st);
int launch_gemm_scales(const float* absmax, const float* other, float* scales, cudaStream_t st);
int launch_split_rows(const float* X, size_t count, const float* scale, __half* hi, __half* lo, cudaStream_t st);
int launch_split_transpose(const float* X, long R, long Cc, long Rp, const float* scale, __half* hi, __half* lo, cudaStream_t st);
int launch_split_both(const float* X, long R, long Cc, long Rp, const float* scale, __half* hi, __half* lo, __half* thi, __half* tlo,
                      cudaStream_t st);

static bool use_tc_backward() {
  const char* e = dev_env("IADMM_TRAIN_SIMT_GEMM");      // development switch: 1 = fp32 CUDA-core GEMMs in the backward
  return !(e && e[0] == '1');
}

// ------------------------------------------------------------------------------------------------
// flat gradient buffer layout = the state_dict order of models/lstm.py:21-41
// ------------------------------------------------------------------------------------------------
struct GradLayout {
  size_t W[4], U[4], b[4], W_h, b_h, rho, alpha, total;
};
GradLayout grad_layout(int h, int length) {
  GradLayout G;
  size_t o = 0;
  for (int g = 0; g < 4; ++g) {
    G.W[g] = o; o += 2 * (size_t)h;
    G.U[g] = o; o += (size_t)h * h;
    G.b[g] = o; o += h;
  }
  G.W_h = o; o += h;
  G.b_h = o; o += 1;
  G.rho = o; o += length;
  G.alpha = o; o += length;
  G.total = o;
  return G;
}

// ------------------------------------------------------------------------------------------------
// generic fp32 GEMM  C[M,N] = op(A) op(B),  A(m,k) = TA ? A[k*lda+m] : A[m*lda+k],  B(k,n) = TB ? B[n*ldb+k] : B[k*ldb+n]
// 128x128x16 tiles, 8x8 per thread.  Plain GEMM (no fusion): used only by the backward pass.
// ------------------------------------------------------------------------------------------------
template <bool TA, bool TB>
__global__ void __launch_bounds__(256) sgemm_kernel(const float* __restrict__ A, const float* __restrict__ Bm,
                                                    float* __restrict__ C, long M, long N, long K, long lda, long ldb,
                                                    long ldc) {
  __shared__ float As[16][128 + 4];
  __shared__ float Bs[16][128 + 4];
  const long m0 = (long)blockIdx.y * 128, n0 = (long)blockIdx.x * 128;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  for (long k0 = 0; k0 < K; k0 += 16) {
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int idx = tid + e * 256;
      int mm, kk;
      if (TA) { mm = idx % 128; kk = idx / 128; } else { kk = idx % 16; mm = idx / 16; }
      const long m = m0 + mm, k = k0 + kk;
      float v = 0.f;
      if (m < M && k < K) v = TA ? A[k * lda + m] : A[m * lda + k];
      As[kk][mm] = v;
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int idx = tid + e * 256;
      int nn, kk;
      if (TB) { kk = idx % 16; nn = idx / 16; } else { nn = idx % 128; kk = idx / 128; }
      const long n = n0 + nn, k = k0 + kk;
      float v = 0.f;
      if (n < N && k < K) v = TB ? Bm[n * ldb + k] : Bm[k * ldb + n];
      Bs[kk][nn] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[kk][ty * 8]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[kk][ty * 8 + 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 8]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 8 + 4]);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const long m = m0 + ty * 8 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const long n = n0 + tx * 8 + j;
      if (n < N) C[m * ldc + n] = acc[i][j];
    }
  }
}

template <bool TA, bool TB>
static int launch_sgemm(const float* A, const float* Bm, float* C, long M, long N, long K, long lda, long ldb, long ldc,
                        cudaStream_t st) {
  const dim3 grid((unsigned)((N + 127) / 128), (unsigned)((M + 127) / 128));
  sgemm_kernel<TA, TB><<<grid, 256, 0, st>>>(A, Bm, C, M, N, K, lda, ldb, ldc);
  IADMM_LAUNCH_CHECK("sgemm_kernel");
  return IADMM_OK;
}

// ------------------------------------------------------------------------------------------------
// weighted column sums  out[w][c] = sum_r weight_w[r] * M[r,c]   (weight NULL = ones), two deterministic stages
// ------------------------------------------------------------------------------------------------
// rows per partial: 256 at large row counts (bounded partial buffer), down to 32 so that a few thousand rows still
// fill the GPU; a function of the row count only
static int cs_rows_per_part(size_t rows) {
  // ~512 parts: enough CTAs for the partial sums (4 column CTAs each at hidden_dim 800), few enough for the final sum
  size_t r = rows / 512;
  r = (r + 7) / 8 * 8;
  return (int)(r < 32 ? 32 : (r > 512 ? 512 : r));
}

template <int NW>
__global__ void __launch_bounds__(256) colsum_partial_kernel(const float* __restrict__ Mx, long rows, int cols,
                                                             const float* __restrict__ w0, const float* __restrict__ w1,
                                                             const float* __restrict__ w2, float wscale,
                                                             float* __restrict__ part, int rows_per_part) {
  // one thread = four consecutive columns (cols % 4 == 0: 128-bit loads, 8 rows in flight), one CTA row = one part of rows
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
  const long r0 = (long)blockIdx.y * rows_per_part;
  if (c >= cols) return;
  const long r1 = (r0 + rows_per_part < rows) ? r0 + rows_per_part : rows;
  float4 acc[NW];
#pragma unroll
  for (int w = 0; w < NW; ++w) acc[w] = make_float4(0.f, 0.f, 0.f, 0.f);
  const float* ws[3] = {w0, w1, w2};
#pragma unroll 8
  for (long r = r0; r < r1; ++r) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(Mx + r * cols + c));
#pragma unroll
    for (int w = 0; w < NW; ++w) {
      const float f = ws[w] ? __ldg(ws[w] + r) * wscale : 1.0f;
      acc[w].x = fmaf(v.x, f, acc[w].x); acc[w].y = fmaf(v.y, f, acc[w].y);
      acc[w].z = fmaf(v.z, f, acc[w].z); acc[w].w = fmaf(v.w, f, acc[w].w);
    }
  }
#pragma unroll
  for (int w = 0; w < NW; ++w) *reinterpret_cast<float4*>(part + ((size_t)blockIdx.y * NW + w) * cols + c) = acc[w];
}

// out_w[c] = sum over partials (fixed order: four interleaved groups of partials, then ((g0+g1)+g2)+g3).
// block = 64 columns x 4 groups; grid = (ceil(cols/64), nw)
__global__ void __launch_bounds__(256) colsum_final_kernel(const float* __restrict__ part, int nparts, int nw, int cols,
                                                           float* __restrict__ out0, float* __restrict__ out1,
                                                           float* __restrict__ out2) {
  __shared__ float sh[4][64];
  const int t = threadIdx.x & 63, g = threadIdx.x >> 6;
  const int c = blockIdx.x * 64 + t;
  const int w = blockIdx.y;
  float* out = (w == 0) ? out0 : (w == 1) ? out1 : out2;
  float s = 0.f;
  if (c < cols) {
#pragma unroll 8
    for (int p = g; p < nparts; p += 4) s += part[((size_t)p * nw + w) * cols + c];
  }
  sh[g][t] = s;
  __syncthreads();
  if (g == 0 && c < cols) out[c] = ((sh[0][t] + sh[1][t]) + sh[2][t]) + sh[3][t];
}

// ------------------------------------------------------------------------------------------------
// backward of the O(N) tail (models/lstm.py:82-94)
// acc[0] += sum rho_bar over inequality rows, acc[1] += over equality rows, acc[2] += alpha_bar
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) tail_bwd_kernel(const KktDims d, const Sched* __restrict__ sched,
                                                       const float* __restrict__ zl, const float* __restrict__ zu,
                                                       const float* __restrict__ x, const float* __restrict__ y,
                                                       const float* __restrict__ z, const float* __restrict__ xv_o,
                                                       const float* __restrict__ gx_o, const float* __restrict__ gy_o,
                                                       const float* __restrict__ gz_o, const float* __restrict__ gxv_o,
                                                       float* __restrict__ Xbar, float* __restrict__ gx,
                                                       float* __restrict__ gy, float* __restrict__ gz,
                                                       double* __restrict__ acc) {
  __shared__ double sh[3][8];
  const size_t n = d.n, m = d.m, N = n + m;
  const size_t rows = (size_t)d.B * N;
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  double a_ineq = 0.0, a_eq = 0.0, a_alpha = 0.0;
  if (idx < rows) {
    const size_t b = idx / N;
    const int r = (int)(idx - b * N);
    const float gxv = gxv_o ? gxv_o[idx] : 0.f;
    if (r < d.n) {
      const size_t j = b * n + r;
      const float g = gx_o ? gx_o[j] : 0.f;
      Xbar[idx] = gxv + sched->alpha * g;
      gx[j] = sched->one_minus_alpha * g;
      a_alpha = (double)g * (double)(xv_o[idx] - x[j]);
    } else {
      const int i = r - d.n;
      const size_t k = b * m + i;
      const bool eq = i >= d.num_ineq;
      const float rho = eq ? sched->rho_eq : sched->rho_ineq;
      const float inv = eq ? sched->inv_rho_eq : sched->inv_rho_ineq;
      const float yo = y[k], zo = z[k], vn = xv_o[idx];
      const float gyo = gy_o ? gy_o[k] : 0.f, gzo = gz_o ? gz_o[k] : 0.f;
      const float zmid = zo + inv * (vn - yo);
      const float u = zmid + inv * yo;
      const float zuu = zu[k], zll = zl[k];
      const float mn = fminf(u, zuu);
      const float zc = fmaxf(mn, zll);
      // torch.min / torch.max split the gradient evenly on exact ties
      const float gmin = (u < zuu) ? 1.f : ((u == zuu) ? 0.5f : 0.f);
      const float gmax = (mn > zll) ? 1.f : ((mn == zll) ? 0.5f : 0.f);
      double rb = (double)gyo * (double)(zmid - zc);               // y' = y + rho (z~ - z')
      float zt_bar = rho * gyo;
      const float zp_bar = gzo - rho * gyo;
      const float ub = zp_bar * gmin * gmax;                        // z' = clip(u)
      zt_bar += ub;                                                 // u = z~ + y / rho
      float yb = gyo + ub * inv;
      rb += (double)ub * (double)(-yo * inv * inv);
      yb -= zt_bar * inv;                                           // z~ = z + (v' - y) / rho
      rb += (double)zt_bar * (double)(-(vn - yo) * inv * inv);
      Xbar[idx] = gxv + zt_bar * inv;
      gy[k] = yb;
      gz[k] = zt_bar;
      if (eq) a_eq = rb; else a_ineq = rb;
    }
  }
  double vals[3] = {a_ineq, a_eq, a_alpha};
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int q = 0; q < 3; ++q) {
    double v = vals[q];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
    if (lane == 0) sh[q][warp] = v;
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += sh[threadIdx.x][w];
    if (t != 0.0) atomicAdd(acc + threadIdx.x, t);
  }
}

// ------------------------------------------------------------------------------------------------
// backward of the cell non-linearities (models/lstm.py:74-80): D = pre-activation adjoints [rows,4h]
// ------------------------------------------------------------------------------------------------
// One warp per coordinate row.  Besides D and gC the same sweep produces what used to be two more passes over D:
// the per-row dots with the two W rows (the cell's direct xv adjoint and the adjoint of g) and max|D| (the scale of
// the fp16 split of the tensor-core backward GEMMs; atomicMax on the bits of a non-negative float).
__global__ void __launch_bounds__(256) cell_bwd_kernel(const float* __restrict__ gates, const float* __restrict__ C_in,
                                                       const float* __restrict__ wh, const float* __restrict__ Xbar,
                                                       const float* __restrict__ gH_o, const float* __restrict__ gC_o,
                                                       const float* __restrict__ wc, float* __restrict__ D,
                                                       float* __restrict__ gC, float* __restrict__ out0,
                                                       float* __restrict__ out1, float* __restrict__ absmax, long rows, int h) {
  const long r = (long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float xb = Xbar[r];
  const size_t h4 = 4 * (size_t)h;
  float a = 0.f, b = 0.f, mx = 0.f;
  for (int j = lane; j < h; j += 32) {
    const size_t idx = (size_t)r * h + j;
    const float4 g4 = *reinterpret_cast<const float4*>(gates + r * h4 + 4 * (size_t)j);
    const float gi = g4.x, gf = g4.y, go = g4.z, gu = g4.w;
    const float c_in = C_in[idx];
    const float cn = gi * gu + gf * c_in;
    const float tc = tanhf(cn);
    const float hbar = (gH_o ? gH_o[idx] : 0.f) - xb * wh[j];            // s_bar = -Xbar (xv' = xv - s)
    const float obar = hbar * tc;
    const float cbar = (gC_o ? gC_o[idx] : 0.f) + hbar * go * (1.f - tc * tc);
    float4 dd;
    dd.x = cbar * gu * gi * (1.f - gi);
    dd.y = cbar * c_in * gf * (1.f - gf);
    dd.z = obar * go * (1.f - go);
    dd.w = cbar * gi * (1.f - gu * gu);
    *reinterpret_cast<float4*>(D + r * h4 + 4 * (size_t)j) = dd;
    gC[idx] = cbar * gf;
    const float4 w0 = __ldg(reinterpret_cast<const float4*>(wc + 4 * (size_t)j));
    const float4 w1 = __ldg(reinterpret_cast<const float4*>(wc + h4 + 4 * (size_t)j));
    a = fmaf(dd.x, w0.x, a); a = fmaf(dd.y, w0.y, a); a = fmaf(dd.z, w0.z, a); a = fmaf(dd.w, w0.w, a);
    b = fmaf(dd.x, w1.x, b); b = fmaf(dd.y, w1.y, b); b = fmaf(dd.z, w1.z, b); b = fmaf(dd.w, w1.w, b);
    const float m4 = fmaxf(fmaxf(fabsf(dd.x), fabsf(dd.y)), fmaxf(fabsf(dd.z), fabsf(dd.w)));
    if (isfinite(m4)) mx = fmaxf(mx, m4);
  }
  a = warp_sum(a); b = warp_sum(b); mx = warp_max(mx);
  if (lane == 0) {
    out0[r] = a; out1[r] = b;
    atomicMax(reinterpret_cast<int*>(absmax), __float_as_int(mx));
  }
}

// ------------------------------------------------------------------------------------------------
// last vector stage of the step backward: assemble the state adjoints and the rho adjoint of the KKT part
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) step_bwd_final_kernel(const KktDims d, const Sched* __restrict__ sched, float sigma,
                                                             const float* __restrict__ xv, const float* __restrict__ y,
                                                             const float* __restrict__ w_save, const float* __restrict__ gbar,
                                                             const float* __restrict__ wbar, const float* __restrict__ ktw,
                                                             const float* __restrict__ Xbar, const float* __restrict__ xvbar_cell,
                                                             float* __restrict__ gxv, float* __restrict__ gx,
                                                             float* __restrict__ gy, float* __restrict__ gz,
                                                             double* __restrict__ acc) {
  __shared__ double sh[2][8];
  const size_t n = d.n, m = d.m, N = n + m;
  const size_t rows = (size_t)d.B * N;
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  double a_ineq = 0.0, a_eq = 0.0;
  if (idx < rows) {
    const size_t b = idx / N;
    const int r = (int)(idx - b * N);
    gxv[idx] = Xbar[idx] + xvbar_cell[idx] + ktw[idx];
    if (r < d.n) {
      gx[b * n + r] += -sigma * wbar[idx];                          // rhs_1 = sigma x - p
    } else {
      const int i = r - d.n;
      const size_t k = b * m + i;
      const bool eq = i >= d.num_ineq;
      const float inv = eq ? sched->inv_rho_eq : sched->inv_rho_ineq;
      const float wb2 = wbar[idx];
      gz[k] += -wb2;                                                // rhs_2 = z - y / rho
      gy[k] += wb2 * inv;
      const double rb = (double)gbar[idx] * (double)(w_save[idx] * inv * inv)        // g_2 = A0 w_1 - w_2 / rho
                      + (double)wb2 * (double)((xv[idx] - y[k]) * inv * inv);        // w_2 = A0 x~ - (v - y) / rho - z
      if (eq) a_eq = rb; else a_ineq = rb;
    }
  }
  double vals[2] = {a_ineq, a_eq};
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    double v = vals[q];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
    if (lane == 0) sh[q][warp] = v;
  }
  __syncthreads();
  if (threadIdx.x < 2) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += sh[threadIdx.x][w];
    if (t != 0.0) atomicAdd(acc + threadIdx.x, t);
  }
}

// scatter the interleaved parameter adjoints into the flat state_dict-ordered gradient buffer (+=)
__global__ void __launch_bounds__(256) scatter_grads_kernel(int h, int t, const float* __restrict__ u32bar,
                                                            const float* __restrict__ w0bar, const float* __restrict__ w1bar,
                                                            const float* __restrict__ bbar, const float* __restrict__ whbar,
                                                            const float* __restrict__ sbar_sum, const double* __restrict__ acc,
                                                            const Sched* __restrict__ sched, GradLayout G,
                                                            float* __restrict__ flat) {
  const size_t total = (size_t)h * 4 * h;
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < total) {
    const int k = (int)(idx / (4 * (size_t)h));
    const int c = (int)(idx - (size_t)k * 4 * h);
    const int j = c >> 2, g = c & 3;
    flat[G.U[g] + (size_t)k * h + j] += u32bar[idx];
  }
  if (idx < (size_t)4 * h) {
    const int j = (int)idx >> 2, g = (int)idx & 3;
    flat[G.W[g] + j] += w0bar[idx];
    flat[G.W[g] + h + j] += w1bar[idx];
    flat[G.b[g] + j] += bbar[idx];
  }
  if (idx < (size_t)h) flat[G.W_h + idx] += whbar[idx];
  if (idx == 0) {
    flat[G.b_h] += sbar_sum[0];
    const float rho = sched->rho_ineq;                       // rho_t = sigmoid(r_t); equality rows carry 1e3 rho_t
    const double rho_bar = acc[0] + 1000.0 * acc[1];
    flat[G.rho + t] += (float)(rho_bar * (double)rho * (1.0 - (double)rho));
    const double s = 0.5 * (double)sched->alpha;              // alpha_t = 2 sigmoid(a_t)
    flat[G.alpha + t] += (float)(acc[2] * 2.0 * s * (1.0 - s));
  }
}

__global__ void negate_sum_kernel(const float* __restrict__ Xbar, long rows, float* __restrict__ out) {
  // b_h adjoint: sum_r s_bar_r = -sum_r Xbar_r   (single block, deterministic)
  __shared__ double sh[32];
  double a = 0.0;
  for (long r = threadIdx.x; r < rows; r += blockDim.x) a -= (double)Xbar[r];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(kFullMask, a, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = a;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += sh[w];
    out[0] = (float)t;
  }
}

// ------------------------------------------------------------------------------------------------
// workspace of the training entry points
// ------------------------------------------------------------------------------------------------
struct TrainWs {
  KktDims d;
  KktScratch s;
  float *head_part, *zeros, *Xbar, *xvbar_cell, *gbar, *D, *u32bar, *u32bar_part, *cs_part, *w0bar, *w1bar, *bbar, *whbar, *sbar_sum;
  __half *h_hi, *h_lo, *h_hi_out, *h_lo_out;      // tensor-core forward: fp16 / e4m3 images of H (in) and scratch (out)
  __half *d_hi, *d_lo, *dt_hi, *dt_lo, *ht_hi, *ht_lo;   // tensor-core backward GEMM operands (D, D^T, H^T as fp16 hi/lo)
  float *gscal;                                   // [8]: absmax(D), then the scales of gemm_scales_kernel at [4..6]
  long rows_p;                                    // row count padded to 8 (pitch of the transposed operands)
  Sched* zero_sched;
  double* acc;
  int cs_parts, cs_rows;
  size_t bytes;
};

static void plan_train(int B, int n, int m, int num_ineq, int h, void* base, TrainWs* W) {
  W->d = make_kkt_dims_train(B, n, m, num_ineq);
  const size_t rows = (size_t)B * (n + m);
  // sized for every gate mode: the tensor-core images and head slots exist where a tensor-core mode runs at this hidden_dim
  GatePlan tc;
  const bool tc_fwd = plan_gates(IADMM_GATES_TC_3XFP16, h, n, m, 1, 0, true, &tc) == IADMM_OK && tc.path == kGatesTc;
  const int simt_tiles = simt_gate_tiles(h), tc_tiles = tc_fwd ? tc_gate_tiles(h) : 0;
  const int max_tiles = simt_tiles > tc_tiles ? simt_tiles : tc_tiles;
  W->cs_rows = cs_rows_per_part(rows);
  W->cs_parts = (int)((rows + W->cs_rows - 1) / W->cs_rows);
  char* p = static_cast<char*>(base);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return base ? p + o : nullptr; };
  float* kkt = reinterpret_cast<float*>(take(kkt_scratch_floats(W->d) * sizeof(float)));
  if (base) kkt_scratch_carve(W->d, kkt, &W->s);
  W->head_part = reinterpret_cast<float*>(take((size_t)max_tiles * rows * sizeof(float)));
  W->h_hi = W->h_lo = W->h_hi_out = W->h_lo_out = nullptr;
  if (tc_fwd) {
    W->h_hi = reinterpret_cast<__half*>(take(rows * (size_t)h * sizeof(__half)));
    W->h_lo = reinterpret_cast<__half*>(take(tc_lo_bytes((long)rows, h)));
    W->h_hi_out = reinterpret_cast<__half*>(take(rows * (size_t)h * sizeof(__half)));
    W->h_lo_out = reinterpret_cast<__half*>(take(tc_lo_bytes((long)rows, h)));
  }
  W->rows_p = (long)((rows + 7) / 8 * 8);
  W->d_hi = W->d_lo = W->dt_hi = W->dt_lo = W->ht_hi = W->ht_lo = nullptr;
  W->gscal = reinterpret_cast<float*>(take(8 * sizeof(float)));
  if (h % 16 == 0) {
    W->d_hi = reinterpret_cast<__half*>(take(rows * 4 * (size_t)h * sizeof(__half)));
    W->d_lo = reinterpret_cast<__half*>(take(rows * 4 * (size_t)h * sizeof(__half)));
    W->dt_hi = reinterpret_cast<__half*>(take((size_t)W->rows_p * 4 * h * sizeof(__half)));
    W->dt_lo = reinterpret_cast<__half*>(take((size_t)W->rows_p * 4 * h * sizeof(__half)));
    W->ht_hi = reinterpret_cast<__half*>(take((size_t)W->rows_p * h * sizeof(__half)));
    W->ht_lo = reinterpret_cast<__half*>(take((size_t)W->rows_p * h * sizeof(__half)));
  }
  W->zeros = reinterpret_cast<float*>(take(rows * sizeof(float)));
  W->zero_sched = reinterpret_cast<Sched*>(take(sizeof(Sched)));
  W->acc = reinterpret_cast<double*>(take(4 * sizeof(double)));
  W->Xbar = reinterpret_cast<float*>(take(rows * sizeof(float)));
  W->xvbar_cell = reinterpret_cast<float*>(take(rows * sizeof(float)));
  W->gbar = reinterpret_cast<float*>(take(rows * sizeof(float)));
  W->D = reinterpret_cast<float*>(take(rows * 4 * (size_t)h * sizeof(float)));
  W->u32bar = reinterpret_cast<float*>(take((size_t)h * 4 * h * sizeof(float)));
  W->u32bar_part = (h % 16 == 0) ? reinterpret_cast<float*>(take((size_t)kMaxSplitK * h * 4 * h * sizeof(float))) : nullptr;   // split-K partials of U_bar
  W->cs_part = reinterpret_cast<float*>(take((size_t)W->cs_parts * 3 * 4 * h * sizeof(float)));
  W->w0bar = reinterpret_cast<float*>(take((size_t)4 * h * sizeof(float)));
  W->w1bar = reinterpret_cast<float*>(take((size_t)4 * h * sizeof(float)));
  W->bbar = reinterpret_cast<float*>(take((size_t)4 * h * sizeof(float)));
  W->whbar = reinterpret_cast<float*>(take((size_t)h * sizeof(float)));
  W->sbar_sum = reinterpret_cast<float*>(take(4 * sizeof(float)));
  W->bytes = off;
}

// The forward gate contraction + cell of one training iteration (fp32 CUDA cores, or the tensor-core kernel with the state
// converted at the boundary), keeping the gate activations.  C_o must already hold C (the cell kernels update it in place).
// Writes gp.head_slots head partials per row.
static int train_gate_forward(const void* packed_weights, const WeightLayout& L, const TrainWs& W, const float* xv, const float* g,
                              const float* H, float* H_o, float* C_o, float* gates_out, size_t rows, int h, const GatePlan& gp,
                              cudaStream_t st) {
  int rc;
  if (gp.path == kGatesFp32)
    return launch_gates_simt(packed_weights, L, xv, g, H, H_o, C_o, W.head_part, (long)rows, h, st, gates_out);
  prof_begin(kProfTrainGates, st);
  if ((rc = launch_split_state(H, W.h_hi, W.h_lo, (long)rows, h, gp.nprod, st))) return rc;
  if (gp.nprod == 2) IADMM_CUDA(cudaMemsetAsync(W.h_lo_out, 0, tc_lo_bytes((long)rows, h), st));
  if ((rc = launch_gates_tc(packed_weights, L, xv, g, W.h_hi, W.h_lo, W.h_hi_out, W.h_lo_out, H_o, C_o, W.head_part,
                            (long)rows, h, gp, st, gates_out))) return rc;
  prof_end(kProfTrainGates, st);
  return IADMM_OK;
}

}  // namespace iadmm

using namespace iadmm;

extern "C" {

int iadmm_param_count(int h, int length, size_t* count) {
  if (h <= 0 || length <= 0 || !count) IADMM_FAIL(IADMM_ESHAPE, "param_count: h=%d length=%d", h, length);
  *count = grad_layout(h, length).total;
  return IADMM_OK;
}

int iadmm_train_workspace_bytes(int B, int n, int m, int h, size_t* bytes) {
  if (B <= 0 || n <= 0 || m < 0 || h <= 0 || !bytes) IADMM_FAIL(IADMM_ESHAPE, "train_workspace_bytes: B=%d n=%d m=%d h=%d", B, n, m, h);
  TrainWs W;
  plan_train(B, n, m, 0, h, nullptr, &W);
  *bytes = W.bytes;
  return IADMM_OK;
}

int iadmm_step_fwd(const void* packed_weights, const float* Q, const float* p, const float* A0, const float* zl,
                   const float* zu, const float* x, const float* y, const float* z, const float* xv, const float* H,
                   const float* C, float* x_o, float* y_o, float* z_o, float* xv_o, float* H_o, float* C_o,
                   float* g_save, float* w_save, float* gates_save, int B, int n, int num_ineq, int num_eq, int h,
                   int length, int t, float sigma, int mode, void* workspace, size_t workspace_bytes, void* stream) {
  const int m = num_ineq + num_eq;
  if (B <= 0 || n <= 0 || num_ineq < 0 || num_eq < 0 || h <= 0 || t < 0 || t >= length)
    IADMM_FAIL(IADMM_ESHAPE, "step_fwd: B=%d n=%d ineq=%d eq=%d h=%d t=%d length=%d", B, n, num_ineq, num_eq, h, t, length);
  if (B > 65535) IADMM_FAIL(IADMM_ESHAPE, "step_fwd: batch %d > 65535", B);
  if (!packed_weights || !Q || !p || !x || !xv || !H || !C || !x_o || !xv_o || !H_o || !C_o || !g_save || !w_save || !workspace)
    IADMM_FAIL(IADMM_EALIGN, "step_fwd: NULL pointer");            // gates_save may be NULL: activations not kept
  if (h % 4 != 0) IADMM_FAIL(IADMM_ESHAPE, "step_fwd: hidden_dim %% 4 != 0 not supported by the training path");
  int rc = check_device();
  if (rc) return rc;
  GatePlan gp;
  if ((rc = plan_gates(mode, h, n, m, 1, 0, true, &gp))) return rc;
  TrainWs W;
  plan_train(B, n, m, num_ineq, h, workspace, &W);
  if (W.bytes > workspace_bytes) IADMM_FAIL(IADMM_EWORK, "step_fwd: workspace too small: %zu < %zu", workspace_bytes, W.bytes);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const WeightLayout L = weight_layout(h, length);
  const char* wbase = static_cast<const char*>(packed_weights);
  const Sched* sk = reinterpret_cast<const Sched*>(wbase + L.off_sched) + t;
  const float* b_h = reinterpret_cast<const float*>(wbase + L.off_bh);
  const size_t N = (size_t)n + m, rows = (size_t)B * N;
  const size_t fb = sizeof(float);
  IADMM_CUDA(cudaMemcpyAsync(x_o, x, (size_t)B * n * fb, cudaMemcpyDeviceToDevice, st));
  if (m > 0) {
    IADMM_CUDA(cudaMemcpyAsync(y_o, y, (size_t)B * m * fb, cudaMemcpyDeviceToDevice, st));
    IADMM_CUDA(cudaMemcpyAsync(z_o, z, (size_t)B * m * fb, cudaMemcpyDeviceToDevice, st));
  }
  IADMM_CUDA(cudaMemcpyAsync(xv_o, xv, rows * fb, cudaMemcpyDeviceToDevice, st));
  IADMM_CUDA(cudaMemcpyAsync(C_o, C, rows * h * fb, cudaMemcpyDeviceToDevice, st));
  prof_begin(kProfTrainKkt, st);
  if ((rc = launch_kkt_pass1(W.d, Q, A0, xv, x, y, W.s, st))) return rc;
  if ((rc = launch_kkt_combine1(W.d, p, xv, x, y, z, sk, sigma, W.s, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                                nullptr, -1, 0, st))) return rc;
  IADMM_CUDA(cudaMemcpyAsync(w_save, W.s.w, rows * fb, cudaMemcpyDeviceToDevice, st));
  if ((rc = launch_kkt_pass2(W.d, Q, A0, W.s, st))) return rc;
  if ((rc = launch_kkt_combine2(W.d, sk, sigma, W.s, st))) return rc;
  IADMM_CUDA(cudaMemcpyAsync(g_save, W.s.g, rows * fb, cudaMemcpyDeviceToDevice, st));
  prof_end(kProfTrainKkt, st);
  // gate contraction of the forward: fp32 CUDA cores, or the tensor-core kernel (same arithmetic as the solve) with
  // the state converted at the boundary; both keep the gate activations for the backward
  if ((rc = train_gate_forward(packed_weights, L, W, xv, W.s.g, H, H_o, C_o, gates_save, rows, h, gp, st))) return rc;
  return launch_tail(W.d, W.head_part, gp.head_slots, b_h, sk, zl, zu, x_o, y_o, z_o, xv_o, st);
}

int iadmm_step_bwd(const void* packed_weights, const float* Q, const float* p, const float* A0, const float* zl,
                   const float* zu, const float* x, const float* y, const float* z, const float* xv, const float* H,
                   const float* C, const float* xv_o, const float* H_o, const float* g_save, const float* w_save,
                   const float* gates_save, const float* gx_o, const float* gy_o, const float* gz_o, const float* gxv_o,
                   const float* gH_o, const float* gC_o, float* gx, float* gy, float* gz, float* gxv, float* gH, float* gC,
                   float* grad_flat, int B, int n, int num_ineq, int num_eq, int h, int length, int t, float sigma,
                   void* workspace, size_t workspace_bytes, void* stream) {
  (void)p;
  const int m = num_ineq + num_eq;
  if (B <= 0 || n <= 0 || num_ineq < 0 || num_eq < 0 || h <= 0 || t < 0 || t >= length)
    IADMM_FAIL(IADMM_ESHAPE, "step_bwd: B=%d n=%d ineq=%d eq=%d h=%d t=%d length=%d", B, n, num_ineq, num_eq, h, t, length);
  if (!packed_weights || !Q || !x || !xv || !H || !C || !xv_o || !H_o || !g_save || !w_save || !gates_save || !gx || !gxv ||
      !gH || !gC || !grad_flat || !workspace)
    IADMM_FAIL(IADMM_EALIGN, "step_bwd: NULL pointer");
  if (m > 0 && (!gy || !gz || !y || !z || !A0 || !zl || !zu)) IADMM_FAIL(IADMM_EALIGN, "step_bwd: NULL constraint pointer");
  if (h % 4 != 0) IADMM_FAIL(IADMM_ESHAPE, "step_bwd: hidden_dim %% 4 != 0 not supported by the training path");
  int rc = check_device();
  if (rc) return rc;
  TrainWs W;
  plan_train(B, n, m, num_ineq, h, workspace, &W);
  if (W.bytes > workspace_bytes) IADMM_FAIL(IADMM_EWORK, "step_bwd: workspace too small: %zu < %zu", workspace_bytes, W.bytes);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const WeightLayout L = weight_layout(h, length);
  const GradLayout G = grad_layout(h, length);
  const char* wbase = static_cast<const char*>(packed_weights);
  const Sched* sk = reinterpret_cast<const Sched*>(wbase + L.off_sched) + t;
  const float* u32 = reinterpret_cast<const float*>(wbase + L.off_u32);
  const float* wc = reinterpret_cast<const float*>(wbase + L.off_wc);
  const float* wh = reinterpret_cast<const float*>(wbase + L.off_wh);
  const size_t N = (size_t)n + m, rows = (size_t)B * N;
  const int h4 = 4 * h;
  const unsigned row_blocks = (unsigned)((rows + 255) / 256);

  IADMM_CUDA(cudaMemsetAsync(W.zeros, 0, rows * sizeof(float), st));
  IADMM_CUDA(cudaMemsetAsync(W.zero_sched, 0, sizeof(Sched), st));
  IADMM_CUDA(cudaMemsetAsync(W.acc, 0, 4 * sizeof(double), st));

  // 1. tail
  prof_begin(kProfTrainCell, st);
  tail_bwd_kernel<<<row_blocks, 256, 0, st>>>(W.d, sk, zl, zu, x, y, z, xv_o, gx_o, gy_o, gz_o, gxv_o, W.Xbar, gx, gy, gz, W.acc);
  IADMM_LAUNCH_CHECK("tail_bwd_kernel");
  // 2. cell non-linearities -> D, gC
  IADMM_CUDA(cudaMemsetAsync(W.gscal, 0, sizeof(float), st));
  cell_bwd_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(gates_save, C, wh, W.Xbar, gH_o, gC_o, wc, W.D, gC, W.xvbar_cell, W.gbar,
                                                               W.gscal, (long)rows, h);
  IADMM_LAUNCH_CHECK("cell_bwd_kernel");
  // 3. small parameter adjoints: W_h (weights s_bar = -Xbar over H'), b_h, and b, W rows over D
  {
    const dim3 g1((unsigned)cdiv(h / 4, 256), (unsigned)W.cs_parts);
    colsum_partial_kernel<1><<<g1, 256, 0, st>>>(H_o, (long)rows, h, W.Xbar, nullptr, nullptr, -1.0f, W.cs_part, W.cs_rows);
    IADMM_LAUNCH_CHECK("colsum_partial_kernel<1>");
    colsum_final_kernel<<<dim3(cdiv(h, 64), 1), 256, 0, st>>>(W.cs_part, W.cs_parts, 1, h, W.whbar, nullptr, nullptr);
    IADMM_LAUNCH_CHECK("colsum_final_kernel");
    negate_sum_kernel<<<1, 1024, 0, st>>>(W.Xbar, (long)rows, W.sbar_sum);
    IADMM_LAUNCH_CHECK("negate_sum_kernel");
    const dim3 g3((unsigned)cdiv(h4 / 4, 256), (unsigned)W.cs_parts);
    colsum_partial_kernel<3><<<g3, 256, 0, st>>>(W.D, (long)rows, h4, nullptr, xv, g_save, 1.0f, W.cs_part, W.cs_rows);
    IADMM_LAUNCH_CHECK("colsum_partial_kernel<3>");
    colsum_final_kernel<<<dim3(cdiv(h4, 64), 3), 256, 0, st>>>(W.cs_part, W.cs_parts, 3, h4, W.bbar, W.w0bar, W.w1bar);
    IADMM_LAUNCH_CHECK("colsum_final_kernel");
  }
  prof_end(kProfTrainCell, st);
  // 4. (input adjoints of the cell, xv direct and g: produced by cell_bwd_kernel)
  // 5. the two GEMMs: H_bar = D U^T ; U_bar = H^T D
  prof_begin(kProfTrainGemm, st);
  if (use_tc_backward() && h % 16 == 0 && rows / 32 < 65535) {
    // tensor cores, fp16 hi/lo split of D * s_D (s_D from max|D|), U * s_U, H * 2^14: fp32-class products
    const float* wscale = reinterpret_cast<const float*>(wbase + L.off_scale);            // [0] = s_U
    const __half* u32hi = reinterpret_cast<const __half*>(wbase + L.off_u32hi);
    const __half* u32lo = reinterpret_cast<const __half*>(wbase + L.off_u32lo);
    if ((rc = launch_gemm_scales(W.gscal, wscale, W.gscal + 4, st))) return rc;          // [4] s_D, [5] 1/(s_D s_U), [6] 1/(s_D 2^14)
    if (W.rows_p != (long)rows) {        // zero the pitch padding of the transposed operands
      IADMM_CUDA(cudaMemsetAsync(W.dt_hi, 0, (size_t)W.rows_p * h4 * sizeof(__half), st));
      IADMM_CUDA(cudaMemsetAsync(W.dt_lo, 0, (size_t)W.rows_p * h4 * sizeof(__half), st));
      IADMM_CUDA(cudaMemsetAsync(W.ht_hi, 0, (size_t)W.rows_p * h * sizeof(__half), st));
      IADMM_CUDA(cudaMemsetAsync(W.ht_lo, 0, (size_t)W.rows_p * h * sizeof(__half), st));
    }
    if ((rc = launch_split_both(W.D, (long)rows, h4, W.rows_p, W.gscal + 4, W.d_hi, W.d_lo, W.dt_hi, W.dt_lo, st))) return rc;
    if ((rc = launch_split_both(H, (long)rows, h, W.rows_p, nullptr, nullptr, nullptr, W.ht_hi, W.ht_lo, st))) return rc;
    const char* m1 = dev_env("IADMM_GEMM1_MASK");
    const char* m2 = dev_env("IADMM_GEMM2_MASK");
    if ((rc = launch_tc_gemm_nt(W.d_hi, W.d_lo, u32hi, u32lo, gH, W.gscal + 5, (long)rows, h, h4, h4, h4, h, st, 1, nullptr,
                                m1 ? atoi(m1) : 7))) return rc;
    // U_bar = H^T D has 7 x 13 output tiles and K = rows: split K so that the (tile, split) units fill the 148 SMs
    int num_sms = 148;
    if ((rc = device_sm_count(&num_sms))) return rc;
    const int splits = tc_gemm_pick_splits(h, h4, (long)rows, num_sms, kMaxSplitK);
    if ((rc = launch_tc_gemm_nt(W.ht_hi, W.ht_lo, W.dt_hi, W.dt_lo, W.u32bar, W.gscal + 6, h, h4, (long)rows, W.rows_p, W.rows_p,
                                h4, st, splits, W.u32bar_part, m2 ? atoi(m2) : 7))) return rc;
  } else {
    if ((rc = launch_sgemm<false, true>(W.D, u32, gH, (long)rows, h, h4, h4, h4, h, st))) return rc;
    if ((rc = launch_sgemm<true, false>(H, W.D, W.u32bar, h, h4, (long)rows, h, h4, h4, st))) return rc;
  }
  prof_end(kProfTrainGemm, st);
  // 6. KKT adjoint: w_bar = K g_bar (pass 1 with zero rhs), then K^T w_bar (pass 2)
  prof_begin(kProfTrainKkt, st);
  if ((rc = launch_kkt_pass1(W.d, Q, A0, W.gbar, W.zeros, W.zeros, W.s, st))) return rc;
  if ((rc = launch_kkt_combine1(W.d, W.zeros, W.gbar, W.zeros, W.zeros, W.zeros, sk, sigma, W.s, nullptr, nullptr, nullptr,
                                nullptr, nullptr, nullptr, nullptr, -1, 0, st))) return rc;
  if ((rc = launch_kkt_pass2(W.d, Q, A0, W.s, st))) return rc;
  if ((rc = launch_kkt_combine2(W.d, sk, sigma, W.s, st))) return rc;
  prof_end(kProfTrainKkt, st);
  // 7. assemble
  step_bwd_final_kernel<<<row_blocks, 256, 0, st>>>(W.d, sk, sigma, xv, y, w_save, W.gbar, W.s.w, W.s.g, W.Xbar, W.xvbar_cell,
                                                    gxv, gx, gy, gz, W.acc);
  IADMM_LAUNCH_CHECK("step_bwd_final_kernel");
  // 8. parameters
  scatter_grads_kernel<<<(unsigned)(((size_t)h * h4 + 255) / 256), 256, 0, st>>>(h, t, W.u32bar, W.w0bar, W.w1bar, W.bbar,
                                                                                W.whbar, W.sbar_sum, W.acc, sk, G, grad_flat);
  IADMM_LAUNCH_CHECK("scatter_grads_kernel");
  return IADMM_OK;
}

// primal_dual_loss (utils.py:68-71) keeping the residual vectors for the backward
int iadmm_residuals_fwd(const float* x, const float* y, const float* z, const float* Q, const float* p, const float* A0,
                        float* pri, float* dual, float* rp_save, float* rd_save, int B, int n, int m, void* workspace,
                        size_t workspace_bytes, void* stream);

}  // extern "C"

namespace iadmm {

// r_p = A0 x - z, r_d = Q x + p + A0^T y from the pass-1 products
__global__ void __launch_bounds__(256) residual_vectors_kernel(const KktDims d, const float* __restrict__ p,
                                                               const float* __restrict__ z, const KktScratch s,
                                                               float* __restrict__ rp, float* __restrict__ rd) {
  const size_t n = d.n, m = d.m, N = n + m;
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)d.B * N) return;
  const size_t b = idx / N;
  const int r = (int)(idx - b * N);
  if (r < d.n) {
    float aty = 0.f;
    const float* part = s.part_a + b * d.chunks_a * 2 * n;
    for (int c = 0; c < d.sum_a; ++c) aty += part[((size_t)c * 2 + 1) * n + r];
    rd[b * n + r] = __fadd_rn(__fadd_rn(s.qx[b * n + r], p[b * n + r]), aty);
  } else {
    const int i = r - d.n;
    rp[b * m + i] = __fsub_rn(s.ax[b * m + i], z[b * m + i]);
  }
}

// a = gdual / dual * r_d (as w_1), b = gpri / pri * r_p (as w_2); gz = -b
__global__ void __launch_bounds__(256) residual_bwd_seed_kernel(const KktDims d, const float* __restrict__ pri,
                                                                const float* __restrict__ dual, const float* __restrict__ rp,
                                                                const float* __restrict__ rd, const float* __restrict__ gpri,
                                                                const float* __restrict__ gdual, float* __restrict__ w,
                                                                float* __restrict__ gz) {
  const size_t n = d.n, m = d.m, N = n + m;
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)d.B * N) return;
  const size_t b = idx / N;
  const int r = (int)(idx - b * N);
  if (r < d.n) {
    const float dn = dual[b];
    const float gd = gdual ? gdual[b] : 0.f;
    w[idx] = (dn > 0.f) ? gd / dn * rd[b * n + r] : 0.f;       // torch: d||v||/dv = v/||v|| (0 at v = 0)
  } else {
    const int i = r - d.n;
    const float pn = pri[b];
    const float gp = gpri ? gpri[b] : 0.f;
    const float v = (pn > 0.f) ? gp / pn * rp[b * m + i] : 0.f;
    w[idx] = v;
    gz[b * m + i] = -v;
  }
}

__global__ void __launch_bounds__(256) residual_bwd_split_kernel(const KktDims d, const float* __restrict__ g,
                                                                 float* __restrict__ gx, float* __restrict__ gy) {
  const size_t n = d.n, m = d.m, N = n + m;
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)d.B * N) return;
  const size_t b = idx / N;
  const int r = (int)(idx - b * N);
  if (r < d.n) gx[b * n + r] = g[idx];
  else         gy[b * m + (r - d.n)] = g[idx];
}

}  // namespace iadmm

extern "C" {

int iadmm_residuals_train_workspace_bytes(int B, int n, int m, size_t* bytes) {
  if (B <= 0 || n <= 0 || m < 0 || !bytes) IADMM_FAIL(IADMM_ESHAPE, "residuals_train_workspace_bytes: B=%d n=%d m=%d", B, n, m);
  *bytes = kkt_scratch_floats(make_kkt_dims_train(B, n, m, 0)) * sizeof(float) + 1024;
  return IADMM_OK;
}

int iadmm_residuals_fwd(const float* x, const float* y, const float* z, const float* Q, const float* p, const float* A0,
                        float* pri, float* dual, float* rp_save, float* rd_save, int B, int n, int m, void* workspace,
                        size_t workspace_bytes, void* stream) {
  if (B <= 0 || n <= 0 || m < 0 || B > 65535) IADMM_FAIL(IADMM_ESHAPE, "residuals_fwd: B=%d n=%d m=%d", B, n, m);
  if (!x || !Q || !p || !pri || !dual || !rd_save || !workspace) IADMM_FAIL(IADMM_EALIGN, "residuals_fwd: NULL pointer");
  if (m > 0 && (!y || !z || !A0 || !rp_save)) IADMM_FAIL(IADMM_EALIGN, "residuals_fwd: NULL constraint pointer");
  int rc = check_device();
  if (rc) return rc;
  const KktDims d = make_kkt_dims_train(B, n, m, 0);
  if (kkt_scratch_floats(d) * sizeof(float) > workspace_bytes) IADMM_FAIL(IADMM_EWORK, "residuals_fwd: workspace too small");
  KktScratch s;
  kkt_scratch_carve(d, static_cast<float*>(workspace), &s);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if ((rc = launch_kkt_pass1_plain(d, Q, A0, x, y, s, st))) return rc;
  if ((rc = launch_kkt_combine1(d, p, nullptr, x, y, z, nullptr, 0.f, s, pri, dual, nullptr, nullptr, nullptr, nullptr,
                                nullptr, 0, 1, st))) return rc;
  const size_t rows = (size_t)B * (n + m);
  KktDims dv = d;
  dv.sum_a = kkt_sum_chunks(d.chunks_a);           // launch_kkt_combine1 folded the partials into chunk 0
  residual_vectors_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(dv, p, z, s, rp_save, rd_save);
  IADMM_LAUNCH_CHECK("residual_vectors_kernel");
  return IADMM_OK;
}

int iadmm_residuals_bwd(const float* Q, const float* A0, const float* pri, const float* dual, const float* rp_save,
                        const float* rd_save, const float* gpri, const float* gdual, float* gx, float* gy, float* gz, int B,
                        int n, int m, void* workspace, size_t workspace_bytes, void* stream) {
  if (B <= 0 || n <= 0 || m < 0 || B > 65535) IADMM_FAIL(IADMM_ESHAPE, "residuals_bwd: B=%d n=%d m=%d", B, n, m);
  if (!Q || !pri || !dual || !rd_save || !gx || !workspace) IADMM_FAIL(IADMM_EALIGN, "residuals_bwd: NULL pointer");
  if (m > 0 && (!A0 || !rp_save || !gy || !gz)) IADMM_FAIL(IADMM_EALIGN, "residuals_bwd: NULL constraint pointer");
  int rc = check_device();
  if (rc) return rc;
  const KktDims d = make_kkt_dims_train(B, n, m, 0);
  const size_t need = kkt_scratch_floats(d) * sizeof(float) + 1024;
  if (need > workspace_bytes) IADMM_FAIL(IADMM_EWORK, "residuals_bwd: workspace too small");
  KktScratch s;
  kkt_scratch_carve(d, static_cast<float*>(workspace), &s);
  Sched* zero_sched = reinterpret_cast<Sched*>(static_cast<char*>(workspace) + align_up(kkt_scratch_floats(d) * sizeof(float), 256));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  IADMM_CUDA(cudaMemsetAsync(zero_sched, 0, sizeof(Sched), st));
  const size_t rows = (size_t)B * (n + m);
  const unsigned blocks = (unsigned)((rows + 255) / 256);
  residual_bwd_seed_kernel<<<blocks, 256, 0, st>>>(d, pri, dual, rp_save, rd_save, gpri, gdual, s.w, gz);
  IADMM_LAUNCH_CHECK("residual_bwd_seed_kernel");
  // [gx; gy] = [Q^T a + A0^T b ; A0 a]  = K^T [a; b] with sigma = 0 and 1/rho = 0
  if ((rc = launch_kkt_pass2(d, Q, A0, s, st))) return rc;
  if ((rc = launch_kkt_combine2(d, zero_sched, 0.f, s, st))) return rc;
  residual_bwd_split_kernel<<<blocks, 256, 0, st>>>(d, s.g, gx, gy);
  IADMM_LAUNCH_CHECK("residual_bwd_split_kernel");
  return IADMM_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// One whole truncated-BPTT window in a single call (main.py:336-358): TL x (iteration + primal_dual_loss) forward,
// loss = loss_scale * sum_t mean_b (pri_t + dual_t), then the backward sweep -- the same kernels as the per-iteration
// entry points above, launched back to back from C.  The per-iteration autograd path is launch/Python bound at
// small batch (config 3, batch 2: 61 ms of 93 ms per window are host overhead); here the host only enqueues.
// ------------------------------------------------------------------------------------------------
namespace iadmm {

struct WindowWs {
  void* step_ws; size_t step_bytes;
  void* res_ws;  size_t res_bytes;
  float *x, *y, *z, *xv, *H, *C;                 // [TL+1] states each
  float *g_save, *w_save, *gates, *pri, *dual, *rp, *rd;   // [TL] each
  float *adj[2][6];                              // ping-pong adjoints gx gy gz gxv gH gC
  float *rgx, *rgy, *rgz, *seed;
  float *Hs, *Cs;                                // recompute: scratch outputs of the re-run gate kernel
  size_t bytes;
};

static void plan_window(int B, int n, int m, int h, int TL, int flags, void* base, WindowWs* W) {
  const bool recompute = (flags & IADMM_TRAIN_RECOMPUTE_GATES) != 0;
  const size_t N = (size_t)n + m, rows = (size_t)B * N, fb = sizeof(float);
  char* p = static_cast<char*>(base);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return base ? p + o : nullptr; };
  TrainWs T;
  plan_train(B, n, m, 0, h, nullptr, &T);
  W->step_bytes = T.bytes; W->step_ws = take(T.bytes);
  W->res_bytes = kkt_scratch_floats(make_kkt_dims_train(B, n, m, 0)) * fb + 1024; W->res_ws = take(W->res_bytes);
  const size_t S = (size_t)TL + 1;
  W->x = reinterpret_cast<float*>(take(S * B * n * fb));
  W->y = reinterpret_cast<float*>(take(S * B * (m > 0 ? m : 1) * fb));
  W->z = reinterpret_cast<float*>(take(S * B * (m > 0 ? m : 1) * fb));
  W->xv = reinterpret_cast<float*>(take(S * rows * fb));
  W->H = reinterpret_cast<float*>(take(S * rows * h * fb));
  W->C = reinterpret_cast<float*>(take(S * rows * h * fb));
  W->g_save = reinterpret_cast<float*>(take((size_t)TL * rows * fb));
  W->w_save = reinterpret_cast<float*>(take((size_t)TL * rows * fb));
  W->gates = reinterpret_cast<float*>(take((size_t)(recompute ? 1 : TL) * rows * 4 * h * fb));
  W->Hs = recompute ? reinterpret_cast<float*>(take(rows * h * fb)) : nullptr;
  W->Cs = recompute ? reinterpret_cast<float*>(take(rows * h * fb)) : nullptr;
  W->pri = reinterpret_cast<float*>(take((size_t)TL * B * fb));
  W->dual = reinterpret_cast<float*>(take((size_t)TL * B * fb));
  W->rp = reinterpret_cast<float*>(take((size_t)TL * B * (m > 0 ? m : 1) * fb));
  W->rd = reinterpret_cast<float*>(take((size_t)TL * B * n * fb));
  for (int s = 0; s < 2; ++s) {
    W->adj[s][0] = reinterpret_cast<float*>(take((size_t)B * n * fb));
    W->adj[s][1] = reinterpret_cast<float*>(take((size_t)B * (m > 0 ? m : 1) * fb));
    W->adj[s][2] = reinterpret_cast<float*>(take((size_t)B * (m > 0 ? m : 1) * fb));
    W->adj[s][3] = reinterpret_cast<float*>(take(rows * fb));
    W->adj[s][4] = reinterpret_cast<float*>(take(rows * h * fb));
    W->adj[s][5] = reinterpret_cast<float*>(take(rows * h * fb));
  }
  W->rgx = reinterpret_cast<float*>(take((size_t)B * n * fb));
  W->rgy = reinterpret_cast<float*>(take((size_t)B * (m > 0 ? m : 1) * fb));
  W->rgz = reinterpret_cast<float*>(take((size_t)B * (m > 0 ? m : 1) * fb));
  W->seed = reinterpret_cast<float*>(take((size_t)B * fb));
  W->bytes = off;
}

__global__ void __launch_bounds__(256) fill_kernel(float* __restrict__ a, size_t count, float v) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) a[i] = v;
}
// a += b (three small vectors at once)
__global__ void __launch_bounds__(256) add3_kernel(float* __restrict__ a0, const float* __restrict__ b0, size_t c0,
                                                   float* __restrict__ a1, const float* __restrict__ b1, size_t c1,
                                                   float* __restrict__ a2, const float* __restrict__ b2, size_t c2) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < c0) a0[i] = __fadd_rn(a0[i], b0[i]);
  if (i < c1) a1[i] = __fadd_rn(a1[i], b1[i]);
  if (i < c2) a2[i] = __fadd_rn(a2[i], b2[i]);
}
// loss = scale * sum_t ( (1/B) sum_b (pri + dual) ), summed per step in the reference's order (main.py:346-347)
__global__ void __launch_bounds__(256) window_loss_kernel(const float* __restrict__ pri, const float* __restrict__ dual, int TL, int B,
                                                          float scale, float* __restrict__ out) {
  __shared__ double sh[8];
  double total = 0.0;
  for (int t = 0; t < TL; ++t) {
    double s = 0.0;
    for (int b = threadIdx.x; b < B; b += 256) s += (double)__fadd_rn(pri[(size_t)t * B + b], dual[(size_t)t * B + b]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(kFullMask, s, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
      double v = 0.0;
      for (int w = 0; w < 8; ++w) v += sh[w];
      total += v / B * (double)scale;
    }
  }
  if (threadIdx.x == 0) out[0] = (float)total;
}

}  // namespace iadmm

extern "C" {

int iadmm_window_workspace_bytes(int B, int n, int m, int h, int TL, int flags, size_t* bytes) {
  if (B <= 0 || n <= 0 || m < 0 || h <= 0 || TL <= 0 || !bytes)
    IADMM_FAIL(IADMM_ESHAPE, "window_workspace_bytes: B=%d n=%d m=%d h=%d TL=%d", B, n, m, h, TL);
  WindowWs W;
  plan_window(B, n, m, h, TL, flags, nullptr, &W);
  *bytes = W.bytes;
  return IADMM_OK;
}

int iadmm_train_window(const void* packed_weights, const float* Q, const float* p, const float* A0, const float* zl,
                       const float* zu, float* x, float* y, float* z, float* xv, float* H, float* C, float* grad_flat,
                       float* loss_out, int B, int n, int num_ineq, int num_eq, int h, int length, int t0, int TL, float sigma,
                       float loss_scale, int mode, int flags, void* workspace, size_t workspace_bytes, void* stream) {
  const int m = num_ineq + num_eq;
  if (B <= 0 || n <= 0 || num_ineq < 0 || num_eq < 0 || h <= 0 || TL <= 0 || t0 < 0 || t0 + TL > length)
    IADMM_FAIL(IADMM_ESHAPE, "train_window: B=%d n=%d ineq=%d eq=%d h=%d t0=%d TL=%d length=%d", B, n, num_ineq, num_eq, h, t0, TL, length);
  if (!packed_weights || !Q || !p || !x || !xv || !H || !C || !grad_flat || !loss_out || !workspace)
    IADMM_FAIL(IADMM_EALIGN, "train_window: NULL pointer");
  if (m > 0 && (!A0 || !zl || !zu || !y || !z)) IADMM_FAIL(IADMM_EALIGN, "train_window: NULL constraint pointer");
  GatePlan gp;
  int rc = plan_gates(mode, h, n, m, 1, 0, true, &gp);
  if (rc) return rc;
  const bool recompute = (flags & IADMM_TRAIN_RECOMPUTE_GATES) != 0;
  WindowWs W;
  plan_window(B, n, m, h, TL, flags, workspace, &W);
  if (W.bytes > workspace_bytes) IADMM_FAIL(IADMM_EWORK, "train_window: workspace too small: %zu < %zu", workspace_bytes, W.bytes);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t N = (size_t)n + m, rows = (size_t)B * N, fb = sizeof(float);
  const size_t sx = (size_t)B * n, sy = (size_t)B * m, sxv = rows, sH = rows * h, sG = rows * 4 * h;
  // state 0 = the caller's state
  IADMM_CUDA(cudaMemcpyAsync(W.x, x, sx * fb, cudaMemcpyDeviceToDevice, st));
  if (m > 0) {
    IADMM_CUDA(cudaMemcpyAsync(W.y, y, sy * fb, cudaMemcpyDeviceToDevice, st));
    IADMM_CUDA(cudaMemcpyAsync(W.z, z, sy * fb, cudaMemcpyDeviceToDevice, st));
  }
  IADMM_CUDA(cudaMemcpyAsync(W.xv, xv, sxv * fb, cudaMemcpyDeviceToDevice, st));
  IADMM_CUDA(cudaMemcpyAsync(W.H, H, sH * fb, cudaMemcpyDeviceToDevice, st));
  IADMM_CUDA(cudaMemcpyAsync(W.C, C, sH * fb, cudaMemcpyDeviceToDevice, st));
  // ---- forward sweep ----
  for (int t = 0; t < TL; ++t) {
    const size_t a = (size_t)t, b = (size_t)t + 1;
    if ((rc = iadmm_step_fwd(packed_weights, Q, p, A0, zl, zu, W.x + a * sx, W.y + a * sy, W.z + a * sy, W.xv + a * sxv, W.H + a * sH,
                             W.C + a * sH, W.x + b * sx, W.y + b * sy, W.z + b * sy, W.xv + b * sxv, W.H + b * sH, W.C + b * sH,
                             W.g_save + a * sxv, W.w_save + a * sxv, recompute ? nullptr : W.gates + a * sG, B, n, num_ineq, num_eq, h,
                             length, t0 + t, sigma, mode, W.step_ws, W.step_bytes, stream))) return rc;
    if ((rc = iadmm_residuals_fwd(W.x + b * sx, W.y + b * sy, W.z + b * sy, Q, p, A0, W.pri + a * B, W.dual + a * B, W.rp + a * sy,
                                  W.rd + a * sx, B, n, m, W.res_ws, W.res_bytes, stream))) return rc;
  }
  window_loss_kernel<<<1, 256, 0, st>>>(W.pri, W.dual, TL, B, loss_scale, loss_out);
  IADMM_LAUNCH_CHECK("window_loss_kernel");
  // ---- backward sweep ----
  fill_kernel<<<(unsigned)((B + 255) / 256), 256, 0, st>>>(W.seed, (size_t)B, loss_scale / (float)B);
  IADMM_LAUNCH_CHECK("fill_kernel");
  const GradLayout G = grad_layout(h, length);
  IADMM_CUDA(cudaMemsetAsync(grad_flat, 0, G.total * fb, st));
  int cur = 0;
  for (int t = TL - 1; t >= 0; --t) {
    const size_t a = (size_t)t, b = (size_t)t + 1;
    float** gin = W.adj[cur];           // adjoint of state t+1 coming from the future (unset at t = TL-1)
    float** gout = W.adj[cur ^ 1];
    const bool last = (t == TL - 1);
    // adjoint of the loss term of this iteration w.r.t. (x, y, z)_{t+1}
    float* rgx = last ? gin[0] : W.rgx;
    float* rgy = last ? gin[1] : W.rgy;
    float* rgz = last ? gin[2] : W.rgz;
    if ((rc = iadmm_residuals_bwd(Q, A0, W.pri + a * B, W.dual + a * B, W.rp + a * sy, W.rd + a * sx, W.seed, W.seed, rgx, rgy, rgz, B,
                                  n, m, W.res_ws, W.res_bytes, stream))) return rc;
    if (!last) {
      const size_t mx = sx > sy ? sx : sy;
      add3_kernel<<<(unsigned)((mx + 255) / 256), 256, 0, st>>>(gin[0], W.rgx, sx, gin[1], W.rgy, sy, gin[2], W.rgz, sy);
      IADMM_LAUNCH_CHECK("add3_kernel");
    }
    const float* gates_t = W.gates + a * sG;
    if (recompute) {
      // SURVEY section 7 step 6: the gate activations of iteration t are not kept over the window (25.6 MB per instance and
      // iteration at n+m = 2000, hidden_dim 800) but recomputed from the saved H_t, C_t, xv_t and g_t by the SAME kernel the
      // forward ran (bit-identical activations), into one iteration's worth of scratch
      TrainWs T;
      plan_train(B, n, m, num_ineq, h, W.step_ws, &T);
      const WeightLayout Lw = weight_layout(h, length);
      IADMM_CUDA(cudaMemcpyAsync(W.Cs, W.C + a * sH, sH * fb, cudaMemcpyDeviceToDevice, st));
      if ((rc = train_gate_forward(packed_weights, Lw, T, W.xv + a * sxv, W.g_save + a * sxv, W.H + a * sH, W.Hs, W.Cs, W.gates,
                                   rows, h, gp, st))) return rc;
      gates_t = W.gates;
    }
    if ((rc = iadmm_step_bwd(packed_weights, Q, p, A0, zl, zu, W.x + a * sx, W.y + a * sy, W.z + a * sy, W.xv + a * sxv, W.H + a * sH,
                             W.C + a * sH, W.xv + b * sxv, W.H + b * sH, W.g_save + a * sxv, W.w_save + a * sxv, gates_t,
                             gin[0], m > 0 ? gin[1] : nullptr, m > 0 ? gin[2] : nullptr, last ? nullptr : gin[3],
                             last ? nullptr : gin[4], last ? nullptr : gin[5], gout[0], gout[1], gout[2], gout[3], gout[4], gout[5],
                             grad_flat, B, n, num_ineq, num_eq, h, length, t0 + t, sigma, W.step_ws, W.step_bytes, stream))) return rc;
    cur ^= 1;
  }
  // ---- the state leaving the window ----
  const size_t e = (size_t)TL;
  IADMM_CUDA(cudaMemcpyAsync(x, W.x + e * sx, sx * fb, cudaMemcpyDeviceToDevice, st));
  if (m > 0) {
    IADMM_CUDA(cudaMemcpyAsync(y, W.y + e * sy, sy * fb, cudaMemcpyDeviceToDevice, st));
    IADMM_CUDA(cudaMemcpyAsync(z, W.z + e * sy, sy * fb, cudaMemcpyDeviceToDevice, st));
  }
  IADMM_CUDA(cudaMemcpyAsync(xv, W.xv + e * sxv, sxv * fb, cudaMemcpyDeviceToDevice, st));
  IADMM_CUDA(cudaMemcpyAsync(H, W.H + e * sH, sH * fb, cudaMemcpyDeviceToDevice, st));
  IADMM_CUDA(cudaMemcpyAsync(C, W.C + e * sH, sH * fb, cudaMemcpyDeviceToDevice, st));
  return IADMM_OK;
}

}  // extern "C"

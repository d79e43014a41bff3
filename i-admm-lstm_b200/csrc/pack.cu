// Weight packing and the penalty schedule (models/lstm.py:21-41 parameters, :60-63 schedule).
//
// The 16 parameter tensors are re-laid once per weight update into what the kernels stream:
//   * gate matrices interleaved per hidden unit (column 4*j+g, g = i,f,o,u) so one thread / one TMEM
//     column group holds all four pre-activations of a unit;
//   * an fp16 hi/lo split of U * 2^s (s chosen so max|U| * 2^s is in [2^12, 2^13)): the tensor-core
//     path multiplies H_hi U_hi + H_lo U_hi + H_hi U_lo in fp32 accumulators, i.e. ~22-bit operands;
//   * rho_t = sigmoid(rho[t]), 1e3 * rho_t, their reciprocals and alpha_t = 2 sigmoid(alpha[t]),
//     rounded to fp32 after every operation exactly like the reference's tensor ops.
#include "common.cuh"

#include <math.h>
#include <cuda_fp8.h>

namespace iadmm {

WeightLayout weight_layout(int h, int length) {
  WeightLayout L;
  L.h = h; L.length = length;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  const size_t H = (size_t)h;
  L.off_u32   = take(H * 4 * H * sizeof(float));
  L.off_wc    = take(2 * 4 * H * sizeof(float));
  L.off_bias  = take(4 * H * sizeof(float));
  L.off_wh    = take(H * sizeof(float));
  L.off_bh    = take(4 * sizeof(float));
  L.off_sched = take((size_t)length * kSchedStride * sizeof(float));
  L.off_scale = take(4 * sizeof(float));
  L.off_uhi   = take(4 * H * H * sizeof(__half));
  L.off_ulo   = take(4 * H * H * sizeof(__half));
  L.off_u32hi = take(4 * H * H * sizeof(__half));
  L.off_u32lo = take(4 * H * H * sizeof(__half));
  L.off_uq8   = take(4 * H * q8_pitch(h));
  L.off_tilep = take((size_t)((h + 63) / 64) * 832 * sizeof(float));
  L.off_tilep_il = take((size_t)((h + 63) / 64) * 832 * sizeof(float));
  L.off_uhi_il = take((size_t)((h + 7) / 8) * 4 * H * 8 * sizeof(__half));
  L.off_uq8_il = take((size_t)((h + 15) / 16) * 2 * 4 * H * 16);
  L.total = off;
  return L;
}

struct PackSrc {
  const float* W[4];
  const float* U[4];
  const float* b[4];
  const float *W_h, *b_h, *rho, *alpha;
};

__global__ void __launch_bounds__(256) pack_small_kernel(PackSrc S, int h, int length, float* __restrict__ wc,
                                                         float* __restrict__ bias, float* __restrict__ wh,
                                                         float* __restrict__ bh, float* __restrict__ sched,
                                                         float* __restrict__ scale, float* __restrict__ tilep,
                                                         float* __restrict__ tilep_il) {
  const int tid = blockIdx.x * blockDim.x + threadIdx.x;
  const int stride = gridDim.x * blockDim.x;
  // per-tile parameter blocks of the tensor-core gate kernel (zero padded past 4h / h)
  const int tiles = (h + 63) / 64;
  for (int i = tid; i < tiles * 832; i += stride) {
    const int t = i / 832, o = i - t * 832;
    float v = 0.f, vil = 0.f;
    if (o < 768) {
      const int a = o >> 8, c = t * 256 + (o & 255);
      if (c < 4 * h) {
        const int j = c >> 2, g = c & 3;
        v = (a == 0) ? S.W[g][j] : (a == 1) ? S.W[g][h + j] : S.b[g][j];
        const int ci = il_gate_col_inv(c);                  // the column that sits at position c of the row-interleaved order
        const int ji = ci >> 2, gi = ci & 3;
        vil = (a == 0) ? S.W[gi][ji] : (a == 1) ? S.W[gi][h + ji] : S.b[gi][ji];
      }
    } else {
      const int u = t * 64 + (o - 768);
      if (u < h) v = vil = S.W_h[u];
    }
    tilep[i] = v;
    tilep_il[i] = vil;
  }
  for (int i = tid; i < 4 * h; i += stride) {
    const int j = i >> 2, g = i & 3;
    wc[i]         = S.W[g][j];
    wc[4 * h + i] = S.W[g][h + j];
    bias[i]       = S.b[g][j];
  }
  for (int j = tid; j < h; j += stride) wh[j] = S.W_h[j];
  if (tid == 0) { bh[0] = S.b_h[0]; scale[2] = 0.f; }
  for (int t = tid; t < length; t += stride) {
    const float rho = sigmoid_ref(S.rho[t]);
    const float rho_eq = __fmul_rn(rho, 1000.0f);
    const float alpha = __fmul_rn(2.0f, sigmoid_ref(S.alpha[t]));
    float* r = sched + (size_t)t * kSchedStride;
    r[0] = rho;
    r[1] = rho_eq;
    r[2] = __frcp_rn(rho);
    r[3] = __frcp_rn(rho_eq);
    r[4] = alpha;
    r[5] = __fsub_rn(1.0f, alpha);
  }
}

__global__ void __launch_bounds__(256) pack_absmax_kernel(PackSrc S, int h, float* __restrict__ scale) {
  const size_t total = (size_t)4 * h * h;
  float mx = 0.f;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int g = (int)(i / ((size_t)h * h));
    const size_t r = i - (size_t)g * h * h;
    const float v = fabsf(S.U[g][r]);
    if (isfinite(v)) mx = fmaxf(mx, v);
  }
  mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<int*>(scale + 2), __float_as_int(mx));  // mx >= 0
}

__device__ __forceinline__ size_t q8_pitch_dev(int h) { return (size_t)((h + 63) / 64) * 128; }

__device__ __forceinline__ uint8_t to_e4m3(float v) {
  return (uint8_t)__nv_cvt_float_to_fp8(v, __NV_SATFINITE, __NV_E4M3);
}

__global__ void __launch_bounds__(256) pack_u_kernel(PackSrc S, int h, float* __restrict__ u32, __half* __restrict__ uhi,
                                                     __half* __restrict__ ulo, __half* __restrict__ u32hi,
                                                     __half* __restrict__ u32lo, uint8_t* __restrict__ uq8,
                                                     __half* __restrict__ uhi_il, uint8_t* __restrict__ uq8_il,
                                                     float* __restrict__ scale) {
  const float mx = scale[2];
  float us = 1.f;
  if (mx > 0.f) us = exp2f((float)(12 - ilogbf(mx)));
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    scale[0] = us;
    scale[1] = 1.0f / (us * (float)(1 << kHShift));
  }
  const size_t total = (size_t)4 * h * h;
  // one thread per (column c = 4j+g, input unit k); consecutive threads -> consecutive c for the fp32
  // image (row k of u32 is contiguous in c)
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int k = (int)(i / (4 * (size_t)h));
    const int c = (int)(i - (size_t)k * 4 * h);
    const int j = c >> 2, g = c & 3;
    const float v = S.U[g][(size_t)k * h + j];
    u32[i] = v;
    const float vs = v * us;
    const __half hi = __float2half_rn(vs);
    const __half lo = __float2half_rn(vs - __half2float(hi));
    uhi[(size_t)c * h + k] = hi;
    ulo[(size_t)c * h + k] = lo;
    u32hi[i] = hi;
    u32lo[i] = lo;
    uint8_t* q = uq8 + (size_t)c * q8_pitch_dev(h) + (size_t)(k >> 6) * 128 + (k & 63);
    q[0]  = to_e4m3(ldexpf(vs - __half2float(hi), kQ8ULoShift));      // residual
    q[64] = to_e4m3(ldexpf(__half2float(hi), kQ8UHiShift));           // coarse copy
    // row-interleaved images: [K group][gate column in the order of il_gate_col][16 bytes]
    const size_t c4 = (size_t)4 * h;
    const size_t ci = (size_t)il_gate_col(c);
    uhi_il[((size_t)(k >> 3) * c4 + ci) * 8 + (k & 7)] = hi;
    uint8_t* qi = uq8_il + ((size_t)(k >> 4) * 2 * c4 + ci) * 16 + (k & 15);
    qi[0]       = q[0];
    qi[c4 * 16] = q[64];
  }
}

// the packing kernels into an image of layout L (width h); schedule rows are computed from S.rho / S.alpha for t < length
static int launch_pack(const PackSrc& S, int h, int length, const WeightLayout& L, char* base, cudaStream_t st) {
  float* scale = reinterpret_cast<float*>(base + L.off_scale);
  pack_small_kernel<<<cdiv(4 * h > length ? 4 * h : length, 256), 256, 0, st>>>(
      S, h, length, reinterpret_cast<float*>(base + L.off_wc), reinterpret_cast<float*>(base + L.off_bias),
      reinterpret_cast<float*>(base + L.off_wh), reinterpret_cast<float*>(base + L.off_bh),
      reinterpret_cast<float*>(base + L.off_sched), scale, reinterpret_cast<float*>(base + L.off_tilep),
      reinterpret_cast<float*>(base + L.off_tilep_il));
  IADMM_LAUNCH_CHECK("pack_small_kernel");
  const size_t total = (size_t)4 * h * h;
  const int blocks = (int)((total + 255) / 256 > 1184 ? 1184 : (total + 255) / 256);
  pack_absmax_kernel<<<blocks, 256, 0, st>>>(S, h, scale);
  IADMM_LAUNCH_CHECK("pack_absmax_kernel");
  // padding bytes of the packed e4m3 rows (last K block when h % 64 != 0) are read by the K=32 MMAs: keep them zero
  IADMM_CUDA(cudaMemsetAsync(base + L.off_uq8, 0, (size_t)4 * h * q8_pitch(h), st));
  IADMM_CUDA(cudaMemsetAsync(base + L.off_uhi_il, 0, L.total - L.off_uhi_il, st));      // K-group padding of the interleaved images
  pack_u_kernel<<<blocks, 256, 0, st>>>(S, h, reinterpret_cast<float*>(base + L.off_u32),
                                        reinterpret_cast<__half*>(base + L.off_uhi),
                                        reinterpret_cast<__half*>(base + L.off_ulo),
                                        reinterpret_cast<__half*>(base + L.off_u32hi),
                                        reinterpret_cast<__half*>(base + L.off_u32lo),
                                        reinterpret_cast<uint8_t*>(base + L.off_uq8),
                                        reinterpret_cast<__half*>(base + L.off_uhi_il),
                                        reinterpret_cast<uint8_t*>(base + L.off_uq8_il), scale);
  IADMM_LAUNCH_CHECK("pack_u_kernel");
  return IADMM_OK;
}

int pack_weights_impl(const float* const W[4], const float* const U[4], const float* const b[4], const float* W_h,
                      const float* b_h, const float* rho, const float* alpha, int h, int length, void* packed,
                      cudaStream_t st) {
  PackSrc S;
  for (int g = 0; g < 4; ++g) { S.W[g] = W[g]; S.U[g] = U[g]; S.b[g] = b[g]; }
  S.W_h = W_h; S.b_h = b_h; S.rho = rho; S.alpha = alpha;
  return launch_pack(S, h, length, weight_layout(h, length), static_cast<char*>(packed), st);
}

// ------------------------------------------------------------------------------------------------
// zero-padded image for training at hidden_dim % 4 != 0 (train_hidden, common.cuh)
// ------------------------------------------------------------------------------------------------
// The parameter tensors of models/lstm.py:21-41 at width hp, read back from the fp32 sections of an image of width h (exact
// copies) and zero past h.  Per gate g: W_g [2][hp], U_g [hp][hp], b_g [hp]; then W_h [hp], b_h [1].
size_t padded_param_floats(int hp) { return 4 * ((size_t)hp * hp + 3 * (size_t)hp) + hp + 1; }

__global__ void __launch_bounds__(256) unpack_padded_kernel(const float* __restrict__ u32, const float* __restrict__ wc,
                                                            const float* __restrict__ bias, const float* __restrict__ wh,
                                                            const float* __restrict__ bh, int h, int hp, float* __restrict__ out) {
  const size_t H4 = 4 * (size_t)h, per_gate = (size_t)hp * hp + 3 * (size_t)hp, total = 4 * per_gate + hp + 1;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    float v = 0.f;
    if (i < 4 * per_gate) {
      const int g = (int)(i / per_gate);
      size_t o = i - (size_t)g * per_gate;
      if (o < 2 * (size_t)hp) {                                   // W_g row a, unit j
        const int a = (int)(o / hp), j = (int)(o - (size_t)a * hp);
        if (j < h) v = wc[a * H4 + 4 * (size_t)j + g];
      } else if ((o -= 2 * (size_t)hp) < (size_t)hp * hp) {       // U_g [k][j]
        const int k = (int)(o / hp), j = (int)(o - (size_t)k * hp);
        if (k < h && j < h) v = u32[(size_t)k * H4 + 4 * (size_t)j + g];
      } else {                                                    // b_g [j]
        const int j = (int)(o - (size_t)hp * hp);
        if (j < h) v = bias[4 * (size_t)j + g];
      }
    } else if (i < 4 * per_gate + hp) {
      const int j = (int)(i - 4 * per_gate);
      if (j < h) v = wh[j];
    } else {
      v = bh[0];
    }
    out[i] = v;
  }
}

int pack_weights_padded(const void* src, int h, int length, int t_first, int sched_rows, int hp, float* params, void* dst,
                        cudaStream_t st) {
  const WeightLayout Ls = weight_layout(h, length), Ld = weight_layout(hp, sched_rows);
  const char* sb = static_cast<const char*>(src);
  char* db = static_cast<char*>(dst);
  IADMM_CUDA(cudaMemsetAsync(dst, 0, Ld.total, st));       // the alignment gaps, as in a zeroed buffer
  const size_t total = padded_param_floats(hp);
  unpack_padded_kernel<<<(unsigned)((total + 255) / 256 > 1184 ? 1184 : (total + 255) / 256), 256, 0, st>>>(
      reinterpret_cast<const float*>(sb + Ls.off_u32), reinterpret_cast<const float*>(sb + Ls.off_wc),
      reinterpret_cast<const float*>(sb + Ls.off_bias), reinterpret_cast<const float*>(sb + Ls.off_wh),
      reinterpret_cast<const float*>(sb + Ls.off_bh), h, hp, params);
  IADMM_LAUNCH_CHECK("unpack_padded_kernel");
  const size_t per_gate = (size_t)hp * hp + 3 * (size_t)hp;
  PackSrc S;
  for (int g = 0; g < 4; ++g) {
    S.W[g] = params + g * per_gate;
    S.U[g] = S.W[g] + 2 * (size_t)hp;
    S.b[g] = S.U[g] + (size_t)hp * hp;
  }
  S.W_h = params + 4 * per_gate;
  S.b_h = S.W_h + hp;
  S.rho = S.alpha = nullptr;
  int rc = launch_pack(S, hp, 0, Ld, db, st);               // the schedule is copied, not recomputed (the image holds no rho)
  if (rc) return rc;
  IADMM_CUDA(cudaMemcpyAsync(db + Ld.off_sched, sb + Ls.off_sched + (size_t)t_first * kSchedStride * sizeof(float),
                             (size_t)sched_rows * kSchedStride * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return IADMM_OK;
}

// ------------------------------------------------------------------------------------------------
// fp32 <-> fp16 hi/lo images of the hidden state (tensor-core path)
// ------------------------------------------------------------------------------------------------
template <bool Q8>
__global__ void __launch_bounds__(256) split_state_kernel(const float* __restrict__ H, __half* __restrict__ hi,
                                                          __half* __restrict__ lo, size_t count, int h) {
  const float s = (float)(1 << kHShift);
  uint8_t* q8 = reinterpret_cast<uint8_t*>(lo);
  const size_t pitch = q8_pitch_dev(h);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x) {
    const float v = H[i] * s;
    const __half a = __float2half_rn(v);
    hi[i] = a;
    if (Q8) {
      const size_t r = i / h;
      const int k = (int)(i - r * h);
      uint8_t* q = q8 + r * pitch + (size_t)(k >> 6) * 128 + (k & 63);
      q[0]  = to_e4m3(ldexpf(v - __half2float(a), kQ8HLoShift));
      q[64] = to_e4m3(ldexpf(v, kQ8HHiShift));
    } else {
      lo[i] = __float2half_rn(v - __half2float(a));
    }
  }
}

size_t tc_lo_bytes(long rows, int h) {
  const size_t a = (size_t)rows * h * sizeof(__half), b = (size_t)rows * q8_pitch(h);
  return a > b ? a : b;
}

int launch_split_state(const float* H, __half* hi, __half* lo, long rows, int h, int nprod, cudaStream_t st) {
  const size_t count = (size_t)rows * h;
  const size_t blocks = (count + 255) / 256;
  const unsigned grid = (unsigned)(blocks > 148 * 16 ? 148 * 16 : blocks);
  if (nprod == 2) {
    IADMM_CUDA(cudaMemsetAsync(lo, 0, (size_t)rows * q8_pitch(h), st));      // padding of the last K block
    split_state_kernel<true><<<grid, 256, 0, st>>>(H, hi, lo, count, h);
  } else {
    split_state_kernel<false><<<grid, 256, 0, st>>>(H, hi, lo, count, h);
  }
  IADMM_LAUNCH_CHECK("split_state_kernel");
  return IADMM_OK;
}

// ---- row-interleaved images (fused solve, F16F8 mode): hi [h/8][rows_p][8] fp16, q8 [h/16][2][rows_p][16] e4m3 ----
__global__ void __launch_bounds__(256) split_state_il_kernel(const float* __restrict__ H, __half* __restrict__ hi,
                                                             uint8_t* __restrict__ q8, long rows, long rows_p, int h) {
  // one thread per (row, 8-unit group): 32-byte read, one 16-byte fp16 store and two 8-byte e4m3 stores
  const float s = (float)(1 << kHShift);
  const int groups = h / 8;
  const size_t total = (size_t)rows * groups;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int kg = (int)(i / (size_t)rows);                 // consecutive threads -> consecutive rows (coalesced stores)
    const size_t r = i - (size_t)kg * rows;
    const float* src = H + r * h + (size_t)kg * 8;
    __half a[8];
    uint8_t res[8], crs[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const float v = src[u] * s;
      a[u] = __float2half_rn(v);
      res[u] = to_e4m3(ldexpf(v - __half2float(a[u]), kQ8HLoShift));
      crs[u] = to_e4m3(ldexpf(v, kQ8HHiShift));
    }
    *reinterpret_cast<uint4*>(hi + ((size_t)kg * rows_p + r) * 8) = *reinterpret_cast<const uint4*>(a);
    uint8_t* q = q8 + ((size_t)(kg >> 1) * 2 * rows_p + r) * 16 + (kg & 1) * 8;
    *reinterpret_cast<uint2*>(q) = *reinterpret_cast<const uint2*>(res);
    *reinterpret_cast<uint2*>(q + (size_t)rows_p * 16) = *reinterpret_cast<const uint2*>(crs);
  }
}

__global__ void __launch_bounds__(256) c_to_il_kernel(const float* __restrict__ C, float* __restrict__ C_il, long rows,
                                                      long rows_p, int h) {
  const int groups = h / 8;
  const size_t total = (size_t)rows * groups;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int kg = (int)(i / (size_t)rows);
    const size_t r = i - (size_t)kg * rows;
    const float4* src = reinterpret_cast<const float4*>(C + r * h + (size_t)kg * 8);
    float4* dst = reinterpret_cast<float4*>(C_il + ((size_t)kg * rows_p + r) * 8);
    dst[0] = src[0];
    dst[1] = src[1];
  }
}

int launch_split_state_il(const float* H, __half* hi, __half* q8, long rows, int h, cudaStream_t st) {
  const long rows_p = il_rows(rows);
  const size_t total = (size_t)rows * (h / 8);
  const size_t blocks = (total + 255) / 256;
  split_state_il_kernel<<<(unsigned)(blocks > 148 * 32 ? 148 * 32 : blocks), 256, 0, st>>>(
      H, hi, reinterpret_cast<uint8_t*>(q8), rows, rows_p, h);
  IADMM_LAUNCH_CHECK("split_state_il_kernel");
  return IADMM_OK;
}

int launch_c_to_il(const float* C, float* C_il, long rows, int h, cudaStream_t st) {
  const long rows_p = il_rows(rows);
  const size_t total = (size_t)rows * (h / 8);
  const size_t blocks = (total + 255) / 256;
  c_to_il_kernel<<<(unsigned)(blocks > 148 * 32 ? 148 * 32 : blocks), 256, 0, st>>>(C, C_il, rows, rows_p, h);
  IADMM_LAUNCH_CHECK("c_to_il_kernel");
  return IADMM_OK;
}

int launch_zero_state(__half* hi, __half* lo, long rows, int h, int nprod, cudaStream_t st) {
  IADMM_CUDA(cudaMemsetAsync(hi, 0, (size_t)rows * h * sizeof(__half), st));
  IADMM_CUDA(cudaMemsetAsync(lo, 0, nprod == 2 ? (size_t)rows * q8_pitch(h) : (size_t)rows * h * sizeof(__half), st));
  return IADMM_OK;
}

}  // namespace iadmm

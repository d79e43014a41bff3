// Coordinate-wise LSTM cell on the 5th-generation tensor cores (IADMM_GATES_TC_3XFP16 / _1XFP16).
//
// Reference: models/lstm.py:74-80.  The four gate products H_t @ U_{i,f,o,u} over all rows = B*(n+m)
// coordinates are ONE [rows,h] x [h,4h] GEMM with weights shared by every row: the only tensor-core
// shaped work on the path (8*rows*h^2 flop per iteration, >99% of the arithmetic at h=800).
//
// Precision.  The reference computes in fp32 and north_star demands rel <= 1e-4 after K=100, which
// rules out bf16 and makes single-pass tf32/fp16 marginal (SURVEY.md section 0, fact 3).  Both operands
// are therefore split into fp16 hi+lo pairs of power-of-two scaled values (H*2^14, U*2^s), and
//     H U  ~=  (H_hi U_hi + H_lo U_hi + H_hi U_lo) * 2^-(14+s)
// is accumulated in fp32 in tensor memory: ~22-bit operands for 3 MMAs at the fp16 rate (cheaper than
// one tf32 MMA per bit of accuracy, and 4 B/element of operand traffic like fp32).  H is kept in this
// hi/lo form between iterations (written by the epilogue), so nothing is re-split on the fly.
//
// Kernel structure (persistent, one CTA per SM, warp specialised):
//   warp 0      TMA producer   cp.async.bulk.tensor 2D tiles (64B swizzle) of H_hi/H_lo [128 x 32] and
//                              U_hi/U_lo [256 x 32] into a 4..8-stage shared-memory ring (mbarrier tx)
//   warp 1      MMA issuer     one elected lane issues tcgen05.mma.cta_group::1.kind::f16 (M=128,
//                              N=256 = 64 hidden units x 4 interleaved gates, K=16), accumulators in
//                              TMEM, double buffered (2 x 256 columns); tcgen05.commit frees smem
//                              stages and publishes finished accumulators
//   warps 2..9  epilogue       tcgen05.ld 32 columns (= 8 units x 4 gates) per step, add the rank-2
//                              input term and bias, sigmoid/tanh, C and H update, fp16 hi/lo re-split of
//                              H, partial dot with W_h -- the whole cell, fused; overlaps the next
//                              tile's MMAs
// Tiles are ordered unit-tile fastest, so CTAs running concurrently share H row tiles through L2 and H is
// read from HBM once per iteration.
#include "common.cuh"
#include "tc_ptx.cuh"
#include "gate_math.cuh"

#include <stdlib.h>

namespace iadmm {

constexpr int kTcBN = 256;            // gate columns per tile (UMMA N) = 64 hidden units
constexpr int kTcUnits = kTcBN / 4;
constexpr int kTcBK = 32;             // K elements per stage (64-byte swizzled rows of fp16)
constexpr int kTcEpiWarps = 8;
constexpr int kTcThreads = 32 * (2 + kTcEpiWarps);
constexpr int kTcABytes = kTcBM * kTcBK * 2;     // 8 KB
constexpr int kTcBBytes = kTcBN * kTcBK * 2;     // 16 KB
constexpr int kTcChunk = 32;                     // TMEM columns per epilogue step (8 units)

int tc_gate_tiles(int h) { return 4 * cdiv(h, kTcUnits); }   // workspace slots: up to four head partials per unit tile (16-warp epilogue)
size_t tc_state_bytes(long rows, int h) { return (size_t)rows * h * sizeof(__half) * 4; }

// ------------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------------
struct TcParams {
  const float* wc;        // [2][4h]
  const float* bias;      // [4h]
  const float* wh;        // [h]
  const float* scale;     // [4]: [1] = dequant
  const float* tilep;     // [unit_tiles][832] per-tile parameter blocks (W0 | W1 | bias | W_h)
  const float* xv;        // [rows]
  const float* g;         // [rows]
  __half* hout_hi;        // [rows][h]
  __half* hout_lo;        // NPROD==2: two e4m3 arrays, [rows*h] residual then [rows*h] coarse copy
  float*  hout_f32;       // optional
  float*  gates_out;      // optional (training): gate activations [rows][4h], column 4j+g
  float*  C;              // [rows][h] in place
  float*  head_part;      // [2*unit_tiles][rows]
  long rows;
  int  h, unit_tiles, k_blocks, stages, nprod;
  int  skew;              // rotate the unit tiles of a row tile by the row-tile index (see tile_unit)
  int  exp;               // development experiments (IADMM_TC_EXP, row-interleaved kernel only, compiled into the EPI 4 instantiation;
                          // results are garbage): 1 = epilogue reads TMEM only,
                          // 2 = no TMA / MMA, 3 = no global traffic in the epilogue, 4 = no cell math, 5 = all rows alias 1024 rows (no DRAM),
                          // 6 = without the U-rounding correction MMA, 7 = without the H-rounding correction MMA (valid numerics of a
                          // U-correction-only mode: the 1.5-unit candidate of DESIGN.md 6b)
  long num_tiles;
  uint32_t wait_ns;       // suspend-time hint of the mbarrier waits (development switch IADMM_TC_WAIT_NS)
  long rows_p;            // row-interleaved layout (EPI 4): rows rounded up to 128; C, hout_hi, hout_lo are [group][rows_p][..]
  float* c_rm_out;        // row-interleaved layout, last iteration: the caller's row-major C
  size_t q8_pitch;        // bytes per row of the packed e4m3 image (NPROD 2)
};

// The fused LSTM-cell epilogue of one tile, executed by the 8 epilogue warps of a CTA (thread = one
// accumulator lane = one coordinate row; a warp pair splits the tile's 8 column chunks of 8 hidden units).
// Split in two so the C loads are in flight while the warp waits for the accumulator.
constexpr int kChunksPerHalf = kTcBN / kTcChunk / 2;   // 4

template <int NCH = kChunksPerHalf>
struct EpiRowT {
  long row;
  bool row_ok;
  float xr, gr;
  float c[NCH][8];
};
typedef EpiRowT<kChunksPerHalf> EpiRow;

template <bool IL = false, int NCH = kChunksPerHalf, bool ABL = false>
__device__ __forceinline__ void lstm_epilogue_prefetch(const TcParams& P, EpiRowT<NCH>& R, int quarter, int half, int lane, int ut,
                                                       long row_base) {
  const int ex = ABL ? P.exp : 0;        // ablation switches exist only in the EPI 4 instantiation (IADMM_TC_EXP)
  R.row = row_base + quarter * 32 + lane;
  R.row_ok = R.row < P.rows;
  R.xr = R.row_ok ? __ldg(P.xv + R.row) : 0.f;
  R.gr = R.row_ok ? __ldg(P.g + R.row) : 0.f;
#pragma unroll
  for (int cc = 0; cc < NCH; ++cc) {
    const int unit0 = ut * kTcUnits + (half * NCH + cc) * 8;
    if (R.row_ok && unit0 < P.h && ex != 3) {
      if (IL) ld_global_v8(P.C + ((size_t)(unit0 >> 3) * P.rows_p + R.row) * 8, R.c[cc]);
      else    ld_global_v8(P.C + (size_t)((ex == 5) ? (R.row & 1023) : R.row) * P.h + unit0, R.c[cc]);
    } else {
#pragma unroll
      for (int u = 0; u < 8; ++u) R.c[cc][u] = 0.f;
    }
  }
}

template <int NPROD>
__device__ __forceinline__ void lstm_epilogue_tile(const TcParams& P, const EpiRow& R, const float* sp, uint32_t tmem_base, int buf,
                                                   int quarter, int half, int ut, float dequant) {
  float hp = 0.f;
  // with h % 16 == 0 two consecutive 8-unit chunks are written together: 32-byte stores of the fp16 image
  // (one sector, one request) and 16-byte stores of the e4m3 images
  const bool wide = (P.h % 16) == 0;
  uint32_t hi_st[4], lo_st[4], res_st[2], crs_st[2];
#pragma unroll
  for (int cc = 0; cc < kChunksPerHalf; ++cc) {
    const int chunk = half * kChunksPerHalf + cc;
    const int unit0 = ut * kTcUnits + chunk * 8;          // first hidden unit of this chunk
    uint32_t v[32];
    const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(buf * kTcBN + chunk * kTcChunk);
    tc_ld32(taddr, v);
    tc_wait_ld();
    if (R.row_ok && unit0 < P.h) {
      const size_t o = (size_t)R.row * P.h + unit0;
      float cnew[8], hnew[8];
      const float4* w0 = reinterpret_cast<const float4*>(sp + chunk * kTcChunk);
      const float4* w1 = reinterpret_cast<const float4*>(sp + kTcBN + chunk * kTcChunk);
      const float4* bb = reinterpret_cast<const float4*>(sp + 2 * kTcBN + chunk * kTcChunk);
      const float4* wh = reinterpret_cast<const float4*>(sp + 3 * kTcBN + chunk * 8);
      const float4 wh0 = wh[0], wh1 = wh[1];
      const float whv[8] = {wh0.x, wh0.y, wh0.z, wh0.w, wh1.x, wh1.y, wh1.z, wh1.w};
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const float4 a0 = w0[u], a1 = w1[u], ab = bb[u];
        // pre_g = xv*W0 + grad*W1 + (H@U) + b   (models/lstm.py:74-77)
        const float pi = fmaf(__uint_as_float(v[u * 4 + 0]), dequant, fmaf(R.gr, a1.x, fmaf(R.xr, a0.x, ab.x)));
        const float pf = fmaf(__uint_as_float(v[u * 4 + 1]), dequant, fmaf(R.gr, a1.y, fmaf(R.xr, a0.y, ab.y)));
        const float po = fmaf(__uint_as_float(v[u * 4 + 2]), dequant, fmaf(R.gr, a1.z, fmaf(R.xr, a0.z, ab.z)));
        const float pu = fmaf(__uint_as_float(v[u * 4 + 3]), dequant, fmaf(R.gr, a1.w, fmaf(R.xr, a0.w, ab.w)));
        const float gi = sigmoid_fast(pi);
        const float gf = sigmoid_fast(pf);
        const float go = sigmoid_fast(po);
        const float gu = tanh_fast(pu);
        const float cn = __fadd_rn(__fmul_rn(gi, gu), __fmul_rn(gf, R.c[cc][u]));  // lstm.py:78
        const float hn = __fmul_rn(go, tanh_fast(cn));                              // lstm.py:79
        cnew[u] = cn;
        hnew[u] = hn;
        hp = fmaf(hn, whv[u], hp);                                                  // lstm.py:80 (partial)
        if (P.gates_out)      // training forward: keep the activations for the hand-written backward
          *reinterpret_cast<float4*>(P.gates_out + (size_t)R.row * 4 * P.h + 4 * (size_t)(unit0 + u)) = make_float4(gi, gf, go, gu);
      }
      st_global_v8(P.C + o, cnew);
      if (P.hout_f32) st_global_v8(P.hout_f32 + o, hnew);
      uint32_t hi[4], lo[4], res[2], crs[2];
      split_hidden8<NPROD>(hnew, hi, lo, res, crs);
      uint8_t* q8row = reinterpret_cast<uint8_t*>(P.hout_lo) + (size_t)R.row * P.q8_pitch;
      if (!wide) {
        *reinterpret_cast<uint4*>(P.hout_hi + o) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        if (NPROD == 3) *reinterpret_cast<uint4*>(P.hout_lo + o) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        if (NPROD == 2) {
          uint8_t* q = q8row + (size_t)(unit0 >> 6) * 128 + (unit0 & 63);
          *reinterpret_cast<uint2*>(q)      = make_uint2(res[0], res[1]);
          *reinterpret_cast<uint2*>(q + 64) = make_uint2(crs[0], crs[1]);
        }
      } else if ((cc & 1) == 0) {
#pragma unroll
        for (int u = 0; u < 4; ++u) { hi_st[u] = hi[u]; lo_st[u] = lo[u]; }
        res_st[0] = res[0]; res_st[1] = res[1]; crs_st[0] = crs[0]; crs_st[1] = crs[1];
      } else {
        const size_t o2 = o - 8;                           // first unit of the chunk pair (multiple of 16)
        const uint32_t w8[8] = {hi_st[0], hi_st[1], hi_st[2], hi_st[3], hi[0], hi[1], hi[2], hi[3]};
        st_global_v8u(P.hout_hi + o2, w8);
        if (NPROD == 3) {
          const uint32_t l8[8] = {lo_st[0], lo_st[1], lo_st[2], lo_st[3], lo[0], lo[1], lo[2], lo[3]};
          st_global_v8u(P.hout_lo + o2, l8);
        }
        if (NPROD == 2) {
          const int u2 = unit0 - 8;
          uint8_t* q = q8row + (size_t)(u2 >> 6) * 128 + (u2 & 63);
          *reinterpret_cast<uint4*>(q)      = make_uint4(res_st[0], res_st[1], res[0], res[1]);
          *reinterpret_cast<uint4*>(q + 64) = make_uint4(crs_st[0], crs_st[1], crs[0], crs[1]);
        }
      }
    }
  }
  if (R.row_ok) P.head_part[((size_t)ut * 2 + half) * P.rows + R.row] = hp;
}


// Work unit `tile` of the persistent grids -> (row tile rt = tile / unit_tiles, unit tile).  The stride between the tiles of a
// CTA (pair) is the number of CTAs (pairs): with 74 pairs and the 4 unit tiles of hidden_dim 200 / 208 a pair would only ever
// see unit tiles {0, 2} or {1, 3}, and since the last unit tile is ragged (8 / 16 of 64 units: a fraction of the epilogue work)
// the pairs on {0, 2} carried 108 full tiles against 54 + 54 ragged ones on the others and set the kernel's time.  Rotating the
// unit tiles of a row tile by rt hands every pair all unit tiles in turn; the unit tiles of a row tile stay adjacent in the
// schedule, so its operand rows are still fetched from HBM once and hit L2 for the other unit tiles.
__device__ __forceinline__ int tile_unit(long tile, long rt, int unit_tiles, int skew) {
  const int j = (int)(tile - rt * unit_tiles);
  return skew ? (int)((j + rt) % unit_tiles) : j;
}

// ------------------------------------------------------------------------------------------------
// Packed-fp32 epilogue (EPI 1, 2).  Power measurements (profiles/r01_gate_power_experiments.json) show the gate
// kernel to be bound by the 1 kW board power cap, not by a pipe: the MMA main loop alone runs at 1.55 GHz, with the
// cell epilogue the SM clock drops to 1.14 GHz, and the epilogue's ~70 instructions per hidden unit are ~20 % of the
// energy.  sm_100 has two-wide fp32 instructions (fma/mul/add.f32x2 -> FFMA2/FMUL2/FADD2): the pre-activations, the
// activation arguments, the tanh polynomials and the state update of two hidden units are issued as pairs, ~40 %
// fewer instructions for bit-identical results (each lane is the same IEEE operation as the scalar form; the cell
// update c = i*u + f*c stays scalar because ptxas contracts mul.f32x2 + add.f32x2 into FFMA2).
// EPI 2 additionally uses the exp-only tanh (absolute error 3e-7, as in the resident kernel).
// ------------------------------------------------------------------------------------------------
// 1 / (1 + 2^t) for both lanes
__device__ __forceinline__ void rcp1p_ex2_2(u64 t, float& r0, float& r1) {
  float t0, t1;
  upk2(t, t0, t1);
  float d0, d1;
  upk2(add2(pk2(ex2_approx(t0), ex2_approx(t1)), bc2(1.0f)), d0, d1);
  r0 = rcp_approx(d0);
  r1 = rcp_approx(d1);
}
// packed form of split_hidden8 (gate_math.cuh): same roundings lane by lane (the scalings are powers of two, the
// residual s - fp16(s) is exact)
template <int NPROD>
__device__ __forceinline__ void split_hidden8_x2(const u64 (&hn2)[4], uint32_t (&hi)[4], uint32_t (&lo)[4], uint32_t (&res)[2],
                                                 uint32_t (&crs)[2]) {
  const u64 hs2 = bc2((float)(1 << kHShift));
  __nv_fp8x2_storage_t r2[4], c2[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const u64 S = mul2(hn2[u], hs2);
    float s0, s1;
    upk2(S, s0, s1);
    const __half2 hh = __floats2half2_rn(s0, s1);
    hi[u] = *reinterpret_cast<const uint32_t*>(&hh);
    const float2 back = __half22float2(hh);
    u64 D;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(D) : "l"(S), "l"(pk2(back.x, back.y)));
    if (NPROD == 3) {
      float d0, d1;
      upk2(D, d0, d1);
      const __half2 hl = __floats2half2_rn(d0, d1);
      lo[u] = *reinterpret_cast<const uint32_t*>(&hl);
    }
    if (NPROD == 2) {
      float r0, r1, c0, c1;
      upk2(mul2(D, bc2(32.0f)), r0, r1);
      upk2(mul2(S, bc2(0.015625f)), c0, c1);
      r2[u] = __nv_cvt_float2_to_fp8x2(make_float2(r0, r1), __NV_SATFINITE, __NV_E4M3);
      c2[u] = __nv_cvt_float2_to_fp8x2(make_float2(c0, c1), __NV_SATFINITE, __NV_E4M3);
    }
  }
  if (NPROD == 2) {
    res[0] = (uint32_t)r2[0] | ((uint32_t)r2[1] << 16); res[1] = (uint32_t)r2[2] | ((uint32_t)r2[3] << 16);
    crs[0] = (uint32_t)c2[0] | ((uint32_t)c2[1] << 16); crs[1] = (uint32_t)c2[2] | ((uint32_t)c2[3] << 16);
  }
}

// tanh of two values: tanh_fast (FAST = false) or tanh_exp (FAST = true) lane by lane
template <bool FAST>
__device__ __forceinline__ u64 tanh2(float x0, float x1, float big0, float big1) {
  // big0/big1 = 1 - 2/(e^{2x}+1) already evaluated by the caller
  if (FAST) return pk2(big0, big1);
  const u64 X = pk2(x0, x1);
  const u64 T = mul2(X, X);
  u64 Q = fma2(T, bc2(0.016433170300270403f), bc2(-0.052669384762106176f));
  Q = fma2(Q, T, bc2(0.133206865150314f));
  Q = fma2(Q, T, bc2(-0.33332945121698027f));
  float s0, s1;
  upk2(fma2(mul2(X, T), Q, X), s0, s1);
  return pk2((fabsf(x0) < 0.55f) ? s0 : big0, (fabsf(x1) < 0.55f) ? s1 : big1);
}

// the same on packed operands (X = the two arguments, BIG = 1 - 2/(e^{2x}+1) of both): nothing is re-paired
template <bool FAST>
__device__ __forceinline__ u64 tanh2p(u64 X, u64 BIG) {
  if (FAST) return BIG;
  const u64 T = mul2(X, X);
  u64 Q = fma2(T, bc2(0.016433170300270403f), bc2(-0.052669384762106176f));
  Q = fma2(Q, T, bc2(0.133206865150314f));
  Q = fma2(Q, T, bc2(-0.33332945121698027f));
  float s0, s1, x0, x1, b0, b1;
  upk2(fma2(mul2(X, T), Q, X), s0, s1);
  upk2(X, x0, x1);
  upk2(BIG, b0, b1);
  return pk2((fabsf(x0) < 0.55f) ? s0 : b0, (fabsf(x1) < 0.55f) ? s1 : b1);
}

template <int NPROD, bool FAST, bool SAVE, bool IL, int NCH = kChunksPerHalf, bool ABL = false, bool SHR = false>
__device__ __forceinline__ void lstm_epilogue_tile_x2(const TcParams& P, const EpiRowT<NCH>& R, const float* sp, uint32_t tmem_base, int buf,
                                                      int quarter, int half, int ut, float dequant) {
  const int ex = ABL ? P.exp : 0;
  u64 hp2 = 0ull;                                       // (even units, odd units) partial head dots
  const bool wide = (P.h % 16) == 0;
  uint32_t hi_st[4], lo_st[4], res_st[2], crs_st[2];
  const u64 xr2 = bc2(R.xr), gr2 = bc2(R.gr), dq2 = bc2(dequant);
  const float kL = 1.4426950408889634f;
  const u64 k_if = bc2(-kL), k_ou = pk2(-kL, 2.0f * kL), k_t = bc2(2.0f * kL);
  const size_t rowoff = (size_t)((ex == 5) ? (R.row & 1023) : R.row);
#pragma unroll
  for (int cc = 0; cc < NCH; ++cc) {
    const int chunk = half * NCH + cc;
    const int unit0 = ut * kTcUnits + chunk * 8;          // first hidden unit of this chunk
    uint32_t v[32];
    const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(buf * kTcBN + chunk * kTcChunk);
    tc_ld32(taddr, v);
    tc_wait_ld();
    if (R.row_ok && unit0 < P.h) {
      const size_t o = rowoff * P.h + unit0;
      float cnew[8], hnew[8];
      u64 hn2[4];
      const float4* w0 = reinterpret_cast<const float4*>(sp + chunk * kTcChunk);
      const float4* w1 = reinterpret_cast<const float4*>(sp + kTcBN + chunk * kTcChunk);
      const float4* bb = reinterpret_cast<const float4*>(sp + 2 * kTcBN + chunk * kTcChunk);
      const float2* wh = reinterpret_cast<const float2*>(sp + 3 * kTcBN + chunk * 8);
#pragma unroll
      for (int u = 0; u < 8; u += 2) {
        if (ex == 4) {
          cnew[u] = R.c[cc][u] + __uint_as_float(v[u * 4]); hnew[u] = __uint_as_float(v[u * 4 + 1]);
          cnew[u + 1] = R.c[cc][u + 1] + __uint_as_float(v[u * 4 + 4]); hnew[u + 1] = __uint_as_float(v[u * 4 + 5]);
          hn2[u >> 1] = pk2(hnew[u], hnew[u + 1]);
          continue;
        }
        float gi[2], gf[2], gu[2];
        u64 GO;                                          // sigmoid(p_o) of the two units
        if constexpr (IL) {
          // Row-interleaved kernels: the eight accumulator columns of a unit pair arrive as (i0 i1 f0 f1 o0 o1 u0 u1)
          // (il_gate_col, common.cuh), the parameter block in the same order: every pair below is one gate of the two units.
          // Lane by lane the same IEEE operations in the same order as the (i, f) / (o, u) pairing of the row-major kernels.
          const float4 a0 = w0[u], a1 = w1[u], ab = bb[u];                    // columns i0 i1 f0 f1
          const float4 c0 = w0[u + 1], c1 = w1[u + 1], cb = bb[u + 1];        // columns o0 o1 u0 u1
          const int b = u * 4;
          // pre_g = xv*W0 + grad*W1 + (H@U) + b   (models/lstm.py:74-77)
          const u64 PI = fma2(pk2(__uint_as_float(v[b]), __uint_as_float(v[b + 1])), dq2,
                              fma2(gr2, pk2(a1.x, a1.y), fma2(xr2, pk2(a0.x, a0.y), pk2(ab.x, ab.y))));
          const u64 PF = fma2(pk2(__uint_as_float(v[b + 2]), __uint_as_float(v[b + 3])), dq2,
                              fma2(gr2, pk2(a1.z, a1.w), fma2(xr2, pk2(a0.z, a0.w), pk2(ab.z, ab.w))));
          const u64 PO = fma2(pk2(__uint_as_float(v[b + 4]), __uint_as_float(v[b + 5])), dq2,
                              fma2(gr2, pk2(c1.x, c1.y), fma2(xr2, pk2(c0.x, c0.y), pk2(cb.x, cb.y))));
          const u64 PU = fma2(pk2(__uint_as_float(v[b + 6]), __uint_as_float(v[b + 7])), dq2,
                              fma2(gr2, pk2(c1.z, c1.w), fma2(xr2, pk2(c0.z, c0.w), pk2(cb.z, cb.w))));
          u64 RU;                                        // 1/(e^{2 p_u}+1)
          if (SHR) {
            // one reciprocal for the four activations of a unit (gate_math.cuh, gates4_shared_rcp_x2): 4 ex2 + 1 rcp per unit
            float t0, t1;
            upk2(mul2(PI, k_if), t0, t1);
            const u64 A = add2(pk2(ex2_approx(fminf(t0, 30.0f)), ex2_approx(fminf(t1, 30.0f))), bc2(1.0f));
            upk2(mul2(PF, k_if), t0, t1);
            const u64 B = add2(pk2(ex2_approx(fminf(t0, 30.0f)), ex2_approx(fminf(t1, 30.0f))), bc2(1.0f));
            upk2(mul2(PO, k_if), t0, t1);
            const u64 C = add2(pk2(ex2_approx(fminf(t0, 30.0f)), ex2_approx(fminf(t1, 30.0f))), bc2(1.0f));
            upk2(mul2(PU, k_t), t0, t1);
            const u64 D = add2(pk2(ex2_approx(fminf(t0, 30.0f)), ex2_approx(fminf(t1, 30.0f))), bc2(1.0f));
            const u64 AB = mul2(A, B), CD = mul2(C, D);
            float q0, q1;
            upk2(mul2(AB, CD), q0, q1);
            const u64 RR = pk2(rcp_approx(q0), rcp_approx(q1));
            const u64 RAB = mul2(RR, CD), RCD = mul2(RR, AB);
            upk2(mul2(RAB, B), gi[0], gi[1]);
            upk2(mul2(RAB, A), gf[0], gf[1]);
            GO = mul2(RCD, D);
            RU = mul2(RCD, C);
          } else {
            float g0, g1;
            rcp1p_ex2_2(mul2(PI, k_if), gi[0], gi[1]);               // sigmoid(p_i)
            rcp1p_ex2_2(mul2(PF, k_if), gf[0], gf[1]);               // sigmoid(p_f)
            rcp1p_ex2_2(mul2(PO, k_if), g0, g1);                     // sigmoid(p_o)
            GO = pk2(g0, g1);
            rcp1p_ex2_2(mul2(PU, k_t), g0, g1);                      // 1/(e^{2 p_u}+1)
            RU = pk2(g0, g1);
          }
          upk2(tanh2p<FAST>(PU, fma2(RU, bc2(-2.0f), bc2(1.0f))), gu[0], gu[1]);
        } else {
          u64 pif[2], pou[2];
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const float4 a0 = w0[u + j], a1 = w1[u + j], ab = bb[u + j];
            const int b = (u + j) * 4;
            // pre_g = xv*W0 + grad*W1 + (H@U) + b   (models/lstm.py:74-77), gates (i,f) and (o,u) as pairs
            pif[j] = fma2(pk2(__uint_as_float(v[b]), __uint_as_float(v[b + 1])), dq2,
                          fma2(gr2, pk2(a1.x, a1.y), fma2(xr2, pk2(a0.x, a0.y), pk2(ab.x, ab.y))));
            pou[j] = fma2(pk2(__uint_as_float(v[b + 2]), __uint_as_float(v[b + 3])), dq2,
                          fma2(gr2, pk2(a1.z, a1.w), fma2(xr2, pk2(a0.z, a0.w), pk2(ab.z, ab.w))));
          }
          float go[2], bigu[2], pu[2];
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            float ru, po_unused;
            if (SHR) {
              // one reciprocal for the four activations of a unit (gate_math.cuh, gates4_shared_rcp_x2): 4 ex2 + 1 rcp
              float t0, t1, t2, t3, a, b, c, d;
              upk2(mul2(pif[j], k_if), t0, t1);
              upk2(mul2(pou[j], k_ou), t2, t3);
              upk2(add2(pk2(ex2_approx(fminf(t0, 30.0f)), ex2_approx(fminf(t1, 30.0f))), bc2(1.0f)), a, b);
              upk2(add2(pk2(ex2_approx(fminf(t2, 30.0f)), ex2_approx(fminf(t3, 30.0f))), bc2(1.0f)), c, d);
              const float ab = a * b, cd = c * d;
              const float r = rcp_approx(ab * cd);
              float rab, rcd;
              upk2(mul2(bc2(r), pk2(cd, ab)), rab, rcd);
              upk2(mul2(bc2(rab), pk2(b, a)), gi[j], gf[j]);
              upk2(mul2(bc2(rcd), pk2(d, c)), go[j], ru);
            } else {
              rcp1p_ex2_2(mul2(pif[j], k_if), gi[j], gf[j]);           // sigmoid(p_i), sigmoid(p_f)
              rcp1p_ex2_2(mul2(pou[j], k_ou), go[j], ru);              // sigmoid(p_o), 1/(e^{2 p_u}+1)
            }
            upk2(pou[j], po_unused, pu[j]);
            bigu[j] = fmaf(-2.0f, ru, 1.0f);
          }
          upk2(tanh2<FAST>(pu[0], pu[1], bigu[0], bigu[1]), gu[0], gu[1]);
          GO = pk2(go[0], go[1]);
        }
        float cn[2];
#pragma unroll
        for (int j = 0; j < 2; ++j)
          cn[j] = __fadd_rn(__fmul_rn(gi[j], gu[j]), __fmul_rn(gf[j], R.c[cc][u + j]));   // lstm.py:78
        float rt0, rt1;
        const u64 CN = pk2(cn[0], cn[1]);
        rcp1p_ex2_2(mul2(CN, k_t), rt0, rt1);
        u64 HN;                                                                           // lstm.py:79
        if constexpr (IL) {
          HN = mul2(GO, tanh2p<FAST>(CN, fma2(pk2(rt0, rt1), bc2(-2.0f), bc2(1.0f))));
        } else {
          float bt0, bt1;
          upk2(fma2(pk2(rt0, rt1), bc2(-2.0f), bc2(1.0f)), bt0, bt1);
          HN = mul2(GO, tanh2<FAST>(cn[0], cn[1], bt0, bt1));
        }
        upk2(HN, hnew[u], hnew[u + 1]);
        hn2[u >> 1] = HN;
        cnew[u] = cn[0]; cnew[u + 1] = cn[1];
        const float2 whp = wh[u >> 1];
        hp2 = fma2(HN, pk2(whp.x, whp.y), hp2);                                           // lstm.py:80 (partial)
        if (SAVE) {           // training forward: keep the activations for the hand-written backward
          float go_s[2];
          upk2(GO, go_s[0], go_s[1]);
#pragma unroll
          for (int j = 0; j < 2; ++j)
            *reinterpret_cast<float4*>(P.gates_out + (size_t)R.row * 4 * P.h + 4 * (size_t)(unit0 + u + j)) =
                make_float4(gi[j], gf[j], go_s[j], gu[j]);
        }
      }
      if (ex == 3) { hp2 = add2(hp2, pk2(cnew[0] + cnew[7], hnew[3])); continue; }
      uint32_t hi[4], lo[4], res[2], crs[2];
      split_hidden8_x2<NPROD>(hn2, hi, lo, res, crs);
      if (IL) {
        // row-interleaved arrays [8-unit group][row][8]: the 32 rows of a warp are adjacent, every access is whole lines
        const size_t gi = (size_t)(unit0 >> 3) * P.rows_p + R.row;
        st_global_v8(P.C + gi * 8, cnew);
        if (P.c_rm_out) st_global_v8(P.c_rm_out + o, cnew);
        if (P.hout_f32) st_global_v8(P.hout_f32 + o, hnew);
        *reinterpret_cast<uint4*>(P.hout_hi + gi * 8) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        if ((cc & 1) == 0 && unit0 + 8 >= P.h) {
          // hidden_dim % 16 == 8: the last 16-unit group has no second half; its padding bytes are multiplied by the MMAs and
          // are written as zero
          uint8_t* q = reinterpret_cast<uint8_t*>(P.hout_lo) + ((size_t)(unit0 >> 4) * 2 * P.rows_p + R.row) * 16;
          *reinterpret_cast<uint4*>(q)                         = make_uint4(res[0], res[1], 0u, 0u);
          *reinterpret_cast<uint4*>(q + (size_t)P.rows_p * 16) = make_uint4(crs[0], crs[1], 0u, 0u);
        } else if ((cc & 1) == 0) {
          res_st[0] = res[0]; res_st[1] = res[1]; crs_st[0] = crs[0]; crs_st[1] = crs[1];
        } else {
          // e4m3 planes [16-unit group][residual | coarse][row][16]
          uint8_t* q = reinterpret_cast<uint8_t*>(P.hout_lo) + ((size_t)(unit0 >> 4) * 2 * P.rows_p + R.row) * 16;
          *reinterpret_cast<uint4*>(q)                        = make_uint4(res_st[0], res_st[1], res[0], res[1]);
          *reinterpret_cast<uint4*>(q + (size_t)P.rows_p * 16) = make_uint4(crs_st[0], crs_st[1], crs[0], crs[1]);
        }
        continue;
      }
      st_global_v8(P.C + o, cnew);
      if (P.hout_f32) st_global_v8(P.hout_f32 + o, hnew);
      uint8_t* q8row = reinterpret_cast<uint8_t*>(P.hout_lo) + rowoff * P.q8_pitch;
      if (!wide) {
        *reinterpret_cast<uint4*>(P.hout_hi + o) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        if (NPROD == 3) *reinterpret_cast<uint4*>(P.hout_lo + o) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        if (NPROD == 2) {
          uint8_t* q = q8row + (size_t)(unit0 >> 6) * 128 + (unit0 & 63);
          *reinterpret_cast<uint2*>(q)      = make_uint2(res[0], res[1]);
          *reinterpret_cast<uint2*>(q + 64) = make_uint2(crs[0], crs[1]);
        }
      } else if ((cc & 1) == 0) {
#pragma unroll
        for (int u = 0; u < 4; ++u) { hi_st[u] = hi[u]; lo_st[u] = lo[u]; }
        res_st[0] = res[0]; res_st[1] = res[1]; crs_st[0] = crs[0]; crs_st[1] = crs[1];
      } else {
        const size_t o2 = o - 8;                           // first unit of the chunk pair (multiple of 16)
        const uint32_t w8[8] = {hi_st[0], hi_st[1], hi_st[2], hi_st[3], hi[0], hi[1], hi[2], hi[3]};
        st_global_v8u(P.hout_hi + o2, w8);
        if (NPROD == 3) {
          const uint32_t l8[8] = {lo_st[0], lo_st[1], lo_st[2], lo_st[3], lo[0], lo[1], lo[2], lo[3]};
          st_global_v8u(P.hout_lo + o2, l8);
        }
        if (NPROD == 2) {
          const int u2 = unit0 - 8;
          uint8_t* q = q8row + (size_t)(u2 >> 6) * 128 + (u2 & 63);
          *reinterpret_cast<uint4*>(q)      = make_uint4(res_st[0], res_st[1], res[0], res[1]);
          *reinterpret_cast<uint4*>(q + 64) = make_uint4(crs_st[0], crs_st[1], crs[0], crs[1]);
        }
      }
    }
  }
  float hpa, hpb;
  upk2(hp2, hpa, hpb);
  if (R.row_ok) P.head_part[((size_t)ut * (8 / NCH) + half) * P.rows + R.row] = hpa + hpb;   // 2 (NCH 4) or 4 (NCH 2) partials per unit tile
}

// stage this tile's W rows / bias / W_h slice (shared by all rows) into shared memory
__device__ __forceinline__ void stage_tile_params(const TcParams& P, float* sp, int et, int ut) {
  const int h4 = 4 * P.h;
  const int c = ut * kTcBN + et;
  const bool ok = c < h4;
  sp[et]             = ok ? __ldg(P.wc + c) : 0.f;
  sp[kTcBN + et]     = ok ? __ldg(P.wc + h4 + c) : 0.f;
  sp[2 * kTcBN + et] = ok ? __ldg(P.bias + c) : 0.f;
  if (et < kTcUnits) {
    const int u = ut * kTcUnits + et;
    sp[3 * kTcBN + et] = (u < P.h) ? __ldg(P.wh + u) : 0.f;
  }
}

constexpr int kParamFloats = 3 * kTcBN + kTcUnits;

// ================================================================================================
// variant A: one CTA per tile (cta_group::1), tile = 128 rows x 256 gate columns
// ================================================================================================
template <int NPROD>
__global__ void __launch_bounds__(kTcThreads, 1)
gates_tc_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo,
                const TcParams P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // carve: [stages x (A_hi | A_lo | B_hi | B_lo)] | params[2][3*256+64] floats | barriers
  constexpr int kStageBytes = (NPROD == 3) ? 2 * (kTcABytes + kTcBBytes) : (kTcABytes + kTcBBytes);
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int stages = P.stages;
  float* sparam = reinterpret_cast<float*>(smem + (size_t)stages * kStageBytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(sparam + 2 * kParamFloats);
  uint64_t* full_bar = bars;                     // [stages]
  uint64_t* empty_bar = bars + stages;           // [stages]
  uint64_t* tfull_bar = bars + 2 * stages;       // [2]
  uint64_t* tempty_bar = bars + 2 * stages + 2;  // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * stages + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a_hi); tma_prefetch_desc(&map_b_hi);
    if (NPROD == 3) { tma_prefetch_desc(&map_a_lo); tma_prefetch_desc(&map_b_lo); }
    for (int s = 0; s < stages; ++s) { mbar_init(smem_u32(&full_bar[s]), 1); mbar_init(smem_u32(&empty_bar[s]), 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(smem_u32(&tfull_bar[b]), 1); mbar_init(smem_u32(&tempty_bar[b]), kTcEpiWarps); }
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

  const int unit_tiles = P.unit_tiles;
  const int h4 = 4 * P.h;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (long tile = blockIdx.x; tile < P.num_tiles; tile += gridDim.x) {
        const long rt = tile / unit_tiles;
        const int  ut = tile_unit(tile, rt, unit_tiles, P.skew);
        const int row0 = (int)(rt * kTcBM);
        const int col0 = ut * kTcBN;
        for (int kb = 0; kb < P.k_blocks; ++kb) {
          mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1);
          const uint32_t fb = smem_u32(&full_bar[stage]);
          mbar_expect_tx(fb, kStageBytes);
          uint8_t* sbase = smem + (size_t)stage * kStageBytes;
          const int k0 = kb * kTcBK;
          tma_load_2d(smem_u32(sbase), &map_a_hi, fb, k0, row0);
          if (NPROD == 3) {
            tma_load_2d(smem_u32(sbase + kTcABytes), &map_a_lo, fb, k0, row0);
            tma_load_2d(smem_u32(sbase + 2 * kTcABytes), &map_b_hi, fb, k0, col0);
            tma_load_2d(smem_u32(sbase + 2 * kTcABytes + kTcBBytes), &map_b_lo, fb, k0, col0);
          } else {
            tma_load_2d(smem_u32(sbase + kTcABytes), &map_b_hi, fb, k0, col0);
          }
          if (++stage == stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      long it = 0;
      for (long tile = blockIdx.x; tile < P.num_tiles; tile += gridDim.x, ++it) {
        const int ut = tile_unit(tile, tile / unit_tiles, unit_tiles, P.skew);
        const int n_cols = min(kTcBN, h4 - ut * kTcBN);
        const uint32_t idesc = make_idesc_f16(n_cols);
        const int buf = (int)(it & 1);
        const uint32_t use = (uint32_t)(it >> 1);
        mbar_wait(smem_u32(&tempty_bar[buf]), (use & 1) ^ 1);     // epilogue drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(buf * kTcBN);
        uint32_t acc = 0;
        for (int kb = 0; kb < P.k_blocks; ++kb) {
          mbar_wait(smem_u32(&full_bar[stage]), phase);
          tc_fence_after();
          const uint32_t sbase = smem_u32(smem + (size_t)stage * kStageBytes);
          const int k_len = min(kTcBK, P.h - kb * kTcBK);
          const int k_steps = (k_len + kTcUK - 1) / kTcUK;
          for (int ks = 0; ks < k_steps; ++ks) {
            const uint32_t koff = (uint32_t)(ks * kTcUK * 2);      // bytes inside the 64-byte swizzled row
            if (NPROD == 3) {
              const uint64_t a_hi = make_smem_desc_sw64(sbase + koff);
              const uint64_t a_lo = make_smem_desc_sw64(sbase + kTcABytes + koff);
              const uint64_t b_hi = make_smem_desc_sw64(sbase + 2 * kTcABytes + koff);
              const uint64_t b_lo = make_smem_desc_sw64(sbase + 2 * kTcABytes + kTcBBytes + koff);
              tc_mma_f16(d_tmem, a_lo, b_hi, idesc, acc); acc = 1;     // small terms first
              tc_mma_f16(d_tmem, a_hi, b_lo, idesc, 1);
              tc_mma_f16(d_tmem, a_hi, b_hi, idesc, 1);
            } else {
              const uint64_t a_hi = make_smem_desc_sw64(sbase + koff);
              const uint64_t b_hi = make_smem_desc_sw64(sbase + kTcABytes + koff);
              tc_mma_f16(d_tmem, a_hi, b_hi, idesc, acc); acc = 1;
            }
          }
          tc_commit(smem_u32(&empty_bar[stage]));                  // frees the smem stage when the MMAs retire
          if (++stage == stages) { stage = 0; phase ^= 1; }
        }
        tc_commit(smem_u32(&tfull_bar[buf]));                      // accumulator complete
      }
    }
  } else {
    // ===================== epilogue: the LSTM cell =====================
    const int ew = warp - 2;                       // 0..7
    const int quarter = warp & 3;                  // TMEM lane quarter this warp may touch
    const int half = (ew >= 4) ? 1 : 0;            // which half of the tile's column chunks
    const int et = threadIdx.x - 64;               // 0..255
    const float dequant = P.scale[1];
    long it = 0;
    for (long tile = blockIdx.x; tile < P.num_tiles; tile += gridDim.x, ++it) {
      const long rt = tile / unit_tiles;
      const int  ut = tile_unit(tile, rt, unit_tiles, P.skew);
      const int buf = (int)(it & 1);
      const uint32_t use = (uint32_t)(it >> 1);
      float* sp = sparam + buf * kParamFloats;
      stage_tile_params(P, sp, et, ut);
      EpiRow R;
      lstm_epilogue_prefetch(P, R, quarter, half, lane, ut, rt * kTcBM);
      asm volatile("bar.sync 1, %0;" ::"n"(kTcEpiWarps * 32) : "memory");
      mbar_wait(smem_u32(&tfull_bar[buf]), use & 1);
      tc_fence_after();
      lstm_epilogue_tile<NPROD>(P, R, sp, tmem_base, buf, quarter, half, ut, dequant);
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

// ================================================================================================
// variant B: CTA pair (cta_group::2): tile = 256 rows x 256 gate columns over two SMs.  Each CTA loads its
// own 128 rows of H and HALF of the U tile; the leader issues M=256 MMAs that read both halves, so the
// shared-memory traffic per MMA drops from 12 KB to 8 KB per SM and the TMA fill from 48 to 32 KB per
// K-block -- the single-CTA form is shared-memory-bandwidth bound (ncu: tensor pipe 71 % active).
// Barrier protocol: `full` lives in the leader and counts the TMA bytes of BOTH CTAs; `empty` and
// `tmem_full` are signalled in both CTAs by multicast tcgen05.commit; `tmem_empty` lives in the leader and
// collects the epilogue warps of both CTAs (the peer's arrive remotely through the cluster window).
// ================================================================================================
// The pair kernel moves 64 K-elements per stage: fp16 operand rows are full 128-byte lines (128B swizzle), the
// e4m3 operand rows 64 bytes (64B swizzle); 3 stages of 64 KB.
constexpr int kPairBK = 64;
constexpr int kPairABytes = kTcBM * kPairBK * 2;          // 16 KB: this CTA's 128 rows of H (fp16)
constexpr int kPairBBytes = (kTcBN / 2) * kPairBK * 2;    // 16 KB: this CTA's half of the U tile (fp16)
constexpr int kPairBBoxRows = 64;                         // U tiles are fetched in 64-row TMA boxes

// CL = cluster size: 2 = one CTA pair; 4 = two pairs working on the SAME unit tile for two different row tiles,
// which lets each 64-row piece of the U tile be fetched from L2 once and multicast to both pairs (the kernel is
// L2->SM fill bound, profiles/README.md): U-tile L2 reads halve, at the price of 132 instead of 148 usable SMs.
// EPI 7: the row-interleaved kernel with SIXTEEN epilogue warps (four per scheduler, two 8-unit chunks per warp and tile) for the
// regime where the cell epilogue, not the MMAs or the power cap, sets the pace (hidden_dim <~ 400: a tile's MMAs take a quarter of
// the time of its epilogue).  20 warps (five per scheduler, so 96 registers per thread; the two-chunk epilogue needs 90): warps 0-3 =
// TMA producer, MMA issuer and two idle warps, warps 4-19 = epilogue (lane quarter = warp % 4).
constexpr int pair_threads(int epi) { return (epi == 7 || epi == 9 || epi == 10) ? 640 : kTcThreads; }
// measured (profiles/r02_epi_warps_sweep.jsonl, same box, gate kernel per launch at the headline problem size): 16 warps win at
// hidden_dim 208 (0.667 vs 0.739 ms), 320 (0.955 vs 1.137), 352 (1.215 vs 1.399) and 384 (1.314 vs 1.510); tie at 400 (1.50);
// 8 warps win from 512 on (2.06 vs 2.13, 640: 3.09 vs 3.11, 800: the power-capped regime)
constexpr int kEpi16MaxHidden = 384;

template <int NPROD, int CL, int EPI>
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(pair_threads(EPI), 1)
gates_tc_pair_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                     const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo,
                     const TcParams P) {
  // NPROD: 3 = fp16 hi/lo split (3 MMAs), 1 = single fp16 MMA, 2 = fp16 MMA + two e4m3 correction MMAs.
  // Stage layout: A_hi16 | A_lo | B_hi16 | B_lo, 16 KB each, every row 128 bytes (128B swizzle).  NPROD 3: lo = fp16
  // residual.  NPROD 2: lo = packed e4m3 image, bytes [0,64) of a row = residual, [64,128) = coarse copy.
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  constexpr bool IL = (EPI >= 4);                     // row-interleaved operands and state (no swizzle); EPI 5: 32-wide K stages, 6: exp-only tanh,
                                                      // 7: 16 epilogue warps
  // The ablation switches of IADMM_TC_EXP (uniform, never-taken branches in production) stay compiled into the 8-warp
  // row-interleaved kernel on purpose: without them ptxas takes 168 instead of 146 registers and schedules the epilogue 3 %
  // slower (same box: 4.74 vs 4.59 ms per launch); declaring a larger block only offers 128 registers with spills.
  constexpr bool ABL = (EPI == 4 || EPI == 8);   // EPI 8: as 4 with one shared reciprocal per unit (measured, not adopted: DESIGN.md)
  const int ex = ABL ? P.exp : 0;
  constexpr bool E16 = (EPI == 7 || EPI == 9 || EPI == 10);                // EPI 9: as 7 with one shared reciprocal per unit; 10: as 9 with the exp-only tanh
  constexpr int kEpiWarps = E16 ? 16 : kTcEpiWarps;
  constexpr int kFirstEpiWarp = E16 ? 4 : 2;
  constexpr int kIlBK = (EPI == 5) ? 32 : 64;
  constexpr uint32_t kIlSub = kIlBK * 256;            // bytes of one operand box: [K groups][128 rows][16 B]
  constexpr int kStageBytes = IL ? 4 * (int)kIlSub : (NPROD == 1) ? (kPairABytes + kPairBBytes) : 2 * (kPairABytes + kPairBBytes);
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // pointer arithmetic keeps the shared address space (LDS, not generic LD)
  const int stages = P.stages;
  float* sparam = reinterpret_cast<float*>(smem + (size_t)stages * kStageBytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(sparam + 2 * kParamFloats);
  uint64_t* full_bar = bars;                     // [stages]   (leader's copy is the live one)
  uint64_t* empty_bar = bars + stages;           // [stages]   both CTAs
  uint64_t* tfull_bar = bars + 2 * stages;       // [2]        both CTAs
  uint64_t* tempty_bar = bars + 2 * stages + 2;  // [2]        leader's copy is the live one
  uint64_t* pfull_bar = bars + 2 * stages + 4;   // [2]        this CTA's parameter block for accumulator buffer b has landed
  uint64_t* pempty_bar = bars + 2 * stages + 6;  // [2]        ... has been consumed by all epilogue warps of this CTA
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * stages + 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = (rank & 1u) == 0;
  const uint32_t leader_rank = rank & ~1u;                 // leader of this CTA's pair
  const uint32_t pair_in_cluster = rank >> 1;
  constexpr int kPairsPerCluster = CL / 2;
  const uint16_t all_mask = (uint16_t)((1u << CL) - 1u);
  const uint16_t pair_mask = (uint16_t)(3u << leader_rank);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a_hi); tma_prefetch_desc(&map_b_hi);
    if (NPROD != 1) { tma_prefetch_desc(&map_a_lo); tma_prefetch_desc(&map_b_lo); }
    // a stage is refilled only after the MMAs of EVERY pair of the cluster have consumed it (multicast writes
    // land in the sibling pair's shared memory too)
    for (int s = 0; s < stages; ++s) { mbar_init(smem_u32(&full_bar[s]), 1); mbar_init(smem_u32(&empty_bar[s]), kPairsPerCluster); }
    for (int b = 0; b < 2; ++b) { mbar_init(smem_u32(&tfull_bar[b]), 1); mbar_init(smem_u32(&tempty_bar[b]), 2 * kEpiWarps); }
    for (int b = 0; b < 2; ++b) { mbar_init(smem_u32(&pfull_bar[b]), 1); mbar_init(smem_u32(&pempty_bar[b]), kEpiWarps); }
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

  const int unit_tiles = P.unit_tiles;
  const int h4 = 4 * P.h;
  // work unit of a cluster = (unit tile, kPairsPerCluster consecutive 256-row tiles); `pair`/`num_pairs` count clusters
  const long pair = blockIdx.x / CL, num_pairs = gridDim.x / CL;

  if (warp < kFirstEpiWarp) {
  if (warp == 0) {
    // ===================== TMA producer (every CTA) =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      constexpr uint32_t kATotal = (NPROD == 1) ? kPairABytes : 2 * kPairABytes;          // bytes of H operands per CTA and stage
      constexpr uint32_t kBBoxTotal = ((NPROD == 1) ? 1 : 2) * kPairBBoxRows * kPairBK * 2; // bytes of one 64-row box of every U operand
      long pit = 0;
      for (long tile = pair; tile < P.num_tiles; tile += num_pairs, ++pit) {
        const long rt = tile / unit_tiles;
        const int  ut = tile_unit(tile, rt, unit_tiles, P.skew);
        // this tile's epilogue parameters: one bulk copy into the buffer of its accumulator (no thread of the epilogue stages
        // anything, no CTA barrier).  Issued after the tile's first operand stages are in flight: the buffer frees up when the
        // epilogue of the tile two back is done, which is also what this tile's MMAs wait for.
        auto stage_params = [&]() {
          const int pb = (int)(pit & 1);
          mbar_wait(smem_u32(&pempty_bar[pb]), (((uint32_t)(pit >> 1)) & 1) ^ 1, P.wait_ns);
          mbar_expect_tx(smem_u32(&pfull_bar[pb]), kParamFloats * 4);
          bulk_load(smem_u32(sparam + pb * kParamFloats), P.tilep + (size_t)ut * kParamFloats, kParamFloats * 4, smem_u32(&pfull_bar[pb]));
        };
        const int kb_count = (ex == 2) ? 0 : P.k_blocks;
        const int kb_params = min(2, kb_count - 1);
        if (kb_count == 0) stage_params();
        const int n_cols = min(kTcBN, h4 - ut * kTcBN);
        const int row0 = (int)((rt * kPairsPerCluster + pair_in_cluster) * (2 * kTcBM)) + (int)(rank & 1u) * kTcBM;   // this CTA's 128 rows of H
        const int col0 = ut * kTcBN + (int)(rank & 1u) * (n_cols / 2);        // first row of this CTA's half of the U tile
        // U boxes are 64 rows.  Full tiles in a 4-CTA cluster: each CTA fetches ONE 64-row piece of its half and
        // multicasts it to the CTA with the same role in the sibling pair.  Otherwise the CTA loads its half itself.
        const bool mcast = (CL == 4) && (n_cols == kTcBN);
        const int  b_boxes = mcast ? 2 : (n_cols / 2 + kPairBBoxRows - 1) / kPairBBoxRows;   // boxes landing in this CTA
        const uint16_t mc_mask = (uint16_t)((1u << rank) | (1u << (rank ^ 2u)));
        for (int kb = 0; kb < kb_count; ++kb) {
          if (kb == kb_params) stage_params();
          mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1, P.wait_ns);
          const uint32_t fb_local = smem_u32(&full_bar[stage]);
          if (leader && !IL) mbar_expect_tx(fb_local, 2u * (kATotal + (uint32_t)b_boxes * kBBoxTotal));   // both CTAs of the pair
          const uint32_t fb = map_to_cta(fb_local, leader_rank);
          uint8_t* sbase = smem + (size_t)stage * kStageBytes;
          const int k0 = kb * kPairBK;
          if (IL) {
            // row-interleaved operands: four boxes per stage, each [K group][128 rows][16 B] (no swizzle)
            if (leader) mbar_expect_tx(fb_local, 2u * 4u * kIlSub);
            const uint32_t sb = smem_u32(sbase);
            tma_load_3d_pair(sb,              &map_a_hi, fb, 0, row0 >> 3, kb * (kIlBK / 8));
            tma_load_4d_pair(sb + kIlSub,     &map_a_lo, fb, 0, row0 >> 3, 0, kb * (kIlBK / 16));
            tma_load_3d_pair(sb + 2 * kIlSub, &map_b_hi, fb, 0, col0 >> 3, kb * (kIlBK / 8));
            tma_load_4d_pair(sb + 3 * kIlSub, &map_b_lo, fb, 0, col0 >> 3, 0, kb * (kIlBK / 16));
            if (++stage == stages) { stage = 0; phase ^= 1; }
            continue;
          }
          auto load_u = [&](const CUtensorMap* map, uint32_t region, int kc) {
            constexpr uint32_t kBoxBytes = kPairBBoxRows * 128;
            if (mcast) {
              const uint32_t q = pair_in_cluster;
              tma_load_2d_pair_mc(region + q * kBoxBytes, map, fb_local, kc, col0 + (int)q * kPairBBoxRows, mc_mask);
            } else {
              for (int bx = 0; bx < b_boxes; ++bx)
                tma_load_2d_pair(region + (uint32_t)bx * kBoxBytes, map, fb, kc, col0 + bx * kPairBBoxRows);
            }
          };
          const uint32_t sb = smem_u32(sbase);
          tma_load_2d_pair(sb, &map_a_hi, fb, k0, row0);
          if (NPROD != 1) {
            // the packed e4m3 tensors are addressed in bytes: K block kb starts at byte kb*128 of a row
            const int k0_lo = (NPROD == 2) ? kb * 128 : k0;
            tma_load_2d_pair(sb + kPairABytes, &map_a_lo, fb, k0_lo, row0);
            load_u(&map_b_hi, sb + 2 * kPairABytes, k0);
            load_u(&map_b_lo, sb + 2 * kPairABytes + kPairBBytes, k0_lo);
          } else {
            load_u(&map_b_hi, sb + kPairABytes, k0);
          }
          if (++stage == stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (leader && lane == 0) {
      int stage = 0; uint32_t phase = 0;
      long it = 0;
      for (long tile = pair; tile < P.num_tiles; tile += num_pairs, ++it) {
        const int ut = tile_unit(tile, tile / unit_tiles, unit_tiles, P.skew);
        const int n_cols = min(kTcBN, h4 - ut * kTcBN);
        const uint32_t idesc = make_idesc_f16(n_cols, 2 * kTcBM);
        const int buf = (int)(it & 1);
        const uint32_t use = (uint32_t)(it >> 1);
        mbar_wait(smem_u32(&tempty_bar[buf]), (use & 1) ^ 1, P.wait_ns);     // both CTAs' epilogues drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(buf * kTcBN);
        uint32_t acc = 0;
        for (int kb = 0; kb < (ex == 2 ? 0 : P.k_blocks); ++kb) {
          mbar_wait(smem_u32(&full_bar[stage]), phase, P.wait_ns);
          tc_fence_after();
          const uint32_t sbase = smem_u32(smem + (size_t)stage * kStageBytes);
          const int k_len = IL ? min(kIlBK, P.h - kb * kIlBK) : min(kPairBK, P.h - kb * kPairBK);
          const int k_steps = (k_len + kTcUK - 1) / kTcUK;
          for (int ks = 0; ks < k_steps; ++ks) {
            const uint32_t koff = (uint32_t)(ks * kTcUK * 2);      // bytes inside the 128-byte swizzled row
            if (IL) {
              // no-swizzle core-matrix tiles: fp16 K-step = two 8-wide K groups 2048 B apart; e4m3 K-step (32 wide) = two
              // 16-wide K groups 4096 B apart, residual plane at +0, coarse plane at +2048
              if ((ks & 1) == 0) {
                const uint32_t a8 = sbase + kIlSub + (uint32_t)(ks >> 1) * 8192, b8 = sbase + 3 * kIlSub + (uint32_t)(ks >> 1) * 8192;
                if (ex != 7) { tc_mma_f8_pair(d_tmem, make_smem_desc_il(a8, 4096), make_smem_desc_il(b8 + 2048, 4096), idesc, acc); acc = 1; }
                if (ex != 6) { tc_mma_f8_pair(d_tmem, make_smem_desc_il(a8 + 2048, 4096), make_smem_desc_il(b8, 4096), idesc, acc); acc = 1; }
              }
              tc_mma_f16_pair(d_tmem, make_smem_desc_il(sbase + (uint32_t)ks * 4096, 2048),
                              make_smem_desc_il(sbase + 2 * kIlSub + (uint32_t)ks * 4096, 2048), idesc, acc);
              acc = 1;
            } else if (NPROD == 3) {
              const uint64_t a_hi = make_smem_desc_sw128(sbase + koff);
              const uint64_t a_lo = make_smem_desc_sw128(sbase + kPairABytes + koff);
              const uint64_t b_hi = make_smem_desc_sw128(sbase + 2 * kPairABytes + koff);
              const uint64_t b_lo = make_smem_desc_sw128(sbase + 2 * kPairABytes + kPairBBytes + koff);
              tc_mma_f16_pair(d_tmem, a_lo, b_hi, idesc, acc); acc = 1;
              tc_mma_f16_pair(d_tmem, a_hi, b_lo, idesc, 1);
              tc_mma_f16_pair(d_tmem, a_hi, b_hi, idesc, 1);
            } else if (NPROD == 2) {
              if ((ks & 1) == 0) {
                // one e4m3 MMA covers 32 K-elements = two fp16 K-steps; residual in bytes [0,64) of the row, coarse in [64,128)
                const uint32_t koff8 = (uint32_t)(ks * kTcUK);
                const uint32_t a8 = sbase + kPairABytes, b8 = sbase + 2 * kPairABytes + kPairBBytes;
                const uint64_t a_res = make_smem_desc_sw128(a8 + koff8);
                const uint64_t a_crs = make_smem_desc_sw128(a8 + 64 + koff8);
                const uint64_t b_res = make_smem_desc_sw128(b8 + koff8);
                const uint64_t b_crs = make_smem_desc_sw128(b8 + 64 + koff8);
                tc_mma_f8_pair(d_tmem, a_res, b_crs, idesc, acc); acc = 1;       // (H - fp16(H)) * U
                tc_mma_f8_pair(d_tmem, a_crs, b_res, idesc, 1);                  // H * (U - fp16(U))
              }
              const uint64_t a_hi = make_smem_desc_sw128(sbase + koff);
              const uint64_t b_hi = make_smem_desc_sw128(sbase + 2 * kPairABytes + koff);
              tc_mma_f16_pair(d_tmem, a_hi, b_hi, idesc, 1);
            } else {
              const uint64_t a_hi = make_smem_desc_sw128(sbase + koff);
              const uint64_t b_hi = make_smem_desc_sw128(sbase + kPairABytes + koff);
              tc_mma_f16_pair(d_tmem, a_hi, b_hi, idesc, acc); acc = 1;
            }
          }
          tc_commit_pair(smem_u32(&empty_bar[stage]), all_mask);   // one of the kPairsPerCluster arrivals, in every CTA
          if (++stage == stages) { stage = 0; phase ^= 1; }
        }
        tc_commit_pair(smem_u32(&tfull_bar[buf]), pair_mask);      // accumulators complete in both CTAs of this pair
      }
    }
  }
  } else {
    // ===================== epilogue (both CTAs, own 128 rows) =====================
    constexpr int NCH = 32 / kEpiWarps;            // 8-unit chunks per warp and tile: 4 (8 warps) or 2 (16 warps)
    const int ew = warp - kFirstEpiWarp;
    const int quarter = warp & 3;
    const int part = ew >> 2;                      // which NCH-chunk slice of the tile's 8 column chunks
    const float dequant = P.scale[1];
    long it = 0;
    for (long tile = pair; tile < P.num_tiles; tile += num_pairs, ++it) {
      const long rt = tile / unit_tiles;
      const int  ut = tile_unit(tile, rt, unit_tiles, P.skew);
      const int buf = (int)(it & 1);
      const uint32_t use = (uint32_t)(it >> 1);
      float* sp = sparam + buf * kParamFloats;
      EpiRowT<NCH> R;
      lstm_epilogue_prefetch<IL, NCH, ABL>(P, R, quarter, part, lane, ut,
                                      (rt * kPairsPerCluster + pair_in_cluster) * (2 * kTcBM) + (long)(rank & 1u) * kTcBM);
      mbar_wait(smem_u32(&pfull_bar[buf]), use & 1, P.wait_ns);      // parameter block (bulk copy issued by the producer warp)
      mbar_wait(smem_u32(&tfull_bar[buf]), use & 1, P.wait_ns);
      tc_fence_after();
      if (ex == 1) {
        uint32_t v[32];
        tc_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(buf * kTcBN + part * NCH * kTcChunk), v);
        tc_wait_ld();
      } else if (EPI == 0) {
        if constexpr (NCH == kChunksPerHalf) lstm_epilogue_tile<NPROD>(P, R, sp, tmem_base, buf, quarter, part, ut, dequant);
      } else {
        lstm_epilogue_tile_x2<NPROD, EPI == 2 || EPI == 6 || EPI == 10, EPI == 3, IL, NCH, ABL, EPI == 8 || EPI == 9 || EPI == 10>(P, R, sp, tmem_base, buf, quarter, part, ut, dequant);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(smem_u32(&pempty_bar[buf]));
        mbar_arrive_cluster(map_to_cta(smem_u32(&tempty_bar[buf]), leader_rank));
      }
    }
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// tile_unit's rotation is only needed when the grid stride and the number of unit tiles share a factor (74 pairs and the 4 unit
// tiles of hidden_dim 200: every pair would see two of the four unit tiles); otherwise the schedule of rounds 1-2 is kept as
// profiled (hidden_dim 800: 13 unit tiles).  Development switch IADMM_TC_SKEW = 0 / 1 forces it off / on.
static int tile_skew_needed(long stride, int unit_tiles, int h) {
  if (const char* e = dev_env("IADMM_TC_SKEW")) return atoi(e) != 0;
  if (h % kTcUnits == 0) return 0;                 // no ragged unit tile: all tiles cost the same
  long a = stride, b = unit_tiles;
  while (b) { const long t = a % b; a = b; b = t; }
  return a > 1;
}

// 2D row-major [rows_total][h] tensor of fp16 (elem_bytes 2, 64B swizzle) or e4m3 bytes (elem_bytes 1, 32B
// swizzle), box = [box_rows][32 elements], OOB reads as zero
int make_map(CUtensorMap* map, const void* base, uint64_t rows_total, int h, int box_rows, int elem_bytes, int box_k) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) IADMM_FAIL(IADMM_ECUDA, "cuTensorMapEncodeTiled entry point not available");
  const cuuint64_t dims[2] = {(cuuint64_t)h, (cuuint64_t)rows_total};
  const cuuint64_t strides[1] = {(cuuint64_t)h * (cuuint64_t)elem_bytes};
  const cuuint32_t box[2] = {(cuuint32_t)box_k, (cuuint32_t)box_rows};
  const int row_bytes = box_k * elem_bytes;
  const CUtensorMapSwizzle swz = row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                 : row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(map, elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_UINT8, 2,
                         const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) IADMM_FAIL(IADMM_ECUDA, "cuTensorMapEncodeTiled failed with CUresult %d (rows=%llu h=%d)", (int)r,
                                    (unsigned long long)rows_total, h);
  return IADMM_OK;
}

int make_map_il(CUtensorMap* map, const void* base, uint64_t rows_total, int groups, bool q8, int box_k) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) IADMM_FAIL(IADMM_ECUDA, "cuTensorMapEncodeTiled entry point not available");
  if (rows_total % 8) IADMM_FAIL(IADMM_ESHAPE, "row-interleaved tensor map needs rows %% 8 == 0");
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r;
  if (!q8) {
    const cuuint64_t dims[3] = {64, (cuuint64_t)(rows_total / 8), (cuuint64_t)groups};
    const cuuint64_t strides[2] = {128, (cuuint64_t)rows_total * 16};
    const cuuint32_t box[3] = {64, 16, (cuuint32_t)(box_k / 8)};
    r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  } else {
    const cuuint64_t dims[4] = {128, (cuuint64_t)(rows_total / 8), 2, (cuuint64_t)groups};
    const cuuint64_t strides[3] = {128, (cuuint64_t)rows_total * 16, (cuuint64_t)rows_total * 32};
    const cuuint32_t box[4] = {128, 16, 2, (cuuint32_t)(box_k / 16)};
    r = enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, const_cast<void*>(base), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  }
  if (r != CUDA_SUCCESS) IADMM_FAIL(IADMM_ECUDA, "cuTensorMapEncodeTiled (interleaved) failed with CUresult %d (rows=%llu groups=%d)", (int)r,
                                    (unsigned long long)rows_total, groups);
  return IADMM_OK;
}

// Encoding a tensor map costs a driver call; a K=100 solve would encode 400 of them for the same six (pointer, shape) pairs
// (two ping-pong state images x two operands, two weight images).  Small per-thread cache keyed by everything that goes
// into the encoding; a map only holds the address and the shape, so a hit is valid whatever the buffer contains.
struct MapKey {
  const void* base; uint64_t rows; int a, b, c, kind;
  bool operator==(const MapKey& o) const { return base == o.base && rows == o.rows && a == o.a && b == o.b && c == o.c && kind == o.kind; }
};
struct MapCache {
  static constexpr int kSlots = 16;
  MapKey key[kSlots];
  CUtensorMap map[kSlots];
  int used = 0, next = 0;
};
template <typename MakeFn>
static int cached_map(CUtensorMap* out, const MapKey& k, MakeFn make) {
  static thread_local MapCache cache;
  for (int i = 0; i < cache.used; ++i)
    if (cache.key[i] == k) { *out = cache.map[i]; return IADMM_OK; }
  int rc = make(out);
  if (rc) return rc;
  const int slot = cache.next;
  cache.key[slot] = k; cache.map[slot] = *out;
  cache.next = (cache.next + 1) % MapCache::kSlots;
  if (cache.used < MapCache::kSlots) ++cache.used;
  return IADMM_OK;
}
static int get_map(CUtensorMap* map, const void* base, uint64_t rows_total, int h, int box_rows, int elem_bytes, int box_k) {
  return cached_map(map, MapKey{base, rows_total, h, box_rows, box_k, elem_bytes},
                    [&](CUtensorMap* m) { return make_map(m, base, rows_total, h, box_rows, elem_bytes, box_k); });
}
static int get_map_il(CUtensorMap* map, const void* base, uint64_t rows_total, int groups, bool q8, int box_k) {
  return cached_map(map, MapKey{base, rows_total, groups, q8 ? 1 : 0, box_k, 16},
                    [&](CUtensorMap* m) { return make_map_il(m, base, rows_total, groups, q8, box_k); });
}

// epilogue warps of the row-interleaved kernel: 16 where the cell epilogue paces the kernel (few K blocks per tile), 8 where
// the MMAs and the power cap do (profiles/README.md); development switch IADMM_TC_EPI_WARPS=8|16 overrides
static int select_epi_warps(int h) {
  const char* w = dev_env("IADMM_TC_EPI_WARPS");
  const int env = w ? atoi(w) : 0;
  return (env == 8 || env == 16) ? env : (h <= kEpi16MaxHidden ? 16 : 8);
}

int plan_gates(int mode, int h, int n, int m, int K, int flags, bool training, GatePlan* p) {
  const bool f16f8 = mode == IADMM_GATES_TC_F16F8 || mode == IADMM_GATES_TC_F16F8U;
  const bool tc = f16f8 || mode == IADMM_GATES_TC_3XFP16 || mode == IADMM_GATES_TC_1XFP16;
  if (!tc && mode != IADMM_GATES_SIMT_FP32) {
    if (training) IADMM_FAIL(IADMM_EMODE, "training: unknown gate mode %d", mode);
    IADMM_FAIL(IADMM_EMODE, "unknown gate mode %d", mode);
  }
  *p = GatePlan{kGatesFp32, 0, false, false, 0, simt_gate_tiles(h)};
  // training runs a tensor-core mode at hidden_dim % 8 != 0 on CUDA cores; the solve rejects it
  if (!tc || (training && h % 8 != 0)) return IADMM_OK;
  if (h % 8 != 0) IADMM_FAIL(IADMM_EMODE, "tensor-core gate modes need hidden_dim %% 8 == 0 (got %d)", h);
  p->path = kGatesTc;
  p->nprod = (mode == IADMM_GATES_TC_3XFP16) ? 3 : (mode == IADMM_GATES_TC_1XFP16) ? 1 : 2;
  p->epi_warps = kTcEpiWarps;
  if (training) {
    // both corrections of the F16F8 modes are kept; at hidden_dim % 16 == 8 as the 3-way split, since only the row-interleaved
    // kernels pad the last 16-unit e4m3 group
    if (f16f8 && h % 16 != 0) p->nprod = 3;
  } else {
    // small instances: one persistent CTA per instance keeps the whole iteration on chip (F16F8U runs full F16F8 there)
    const char* res_sw = dev_env("IADMM_RESIDENT");            // development switch: 0 = always the streaming path
    if (!(flags & IADMM_F_STREAMING) && !(res_sw && res_sw[0] == '0') && resident_eligible(n, m, h, p->nprod)) {
      p->path = kGatesResident;
      p->epi_warps = p->head_slots = 0;
      return IADMM_OK;
    }
    // Row-interleaved state for the fused F16F8 solve (K >= 2; a single step would only pay the layout conversion, unless the
    // caller keeps the planes for the next call): the epilogue of the gate kernel then touches whole 128-byte lines instead of
    // one 32-byte sector per row.  With hidden_dim % 16 == 8 only these kernels pad the last 16-unit e4m3 group.
    const char* il_sw = dev_env("IADMM_TC_INTERLEAVED");       // development switch: 0 = row-major state
    const bool keep = (flags & (IADMM_F_KEEP_PLANES | IADMM_F_RESUME)) != 0;
    p->interleaved = f16f8 && (K >= 2 || h % 16 != 0 || keep) && !(il_sw && il_sw[0] == '0');
    if (f16f8 && h % 16 != 0 && !p->interleaved) IADMM_FAIL(IADMM_EMODE, "hidden_dim %% 16 != 0 needs the row-interleaved fp16+fp8 kernels");
    if ((flags & IADMM_F_RESUME) && !p->interleaved)
      IADMM_FAIL(IADMM_EMODE, "solve: IADMM_F_RESUME needs the row-interleaved fp16+fp8 path (iadmm_solve_state_resumable)");
    p->drop_h = p->interleaved && mode == IADMM_GATES_TC_F16F8U;
    // the F16F8U product set and the IADMM_TC_EXP ablations exist only in the 8-warp instantiation
    const char* exp_sw = dev_env("IADMM_TC_EXP");
    if (p->interleaved && !p->drop_h && !(exp_sw && atoi(exp_sw) != 0)) p->epi_warps = select_epi_warps(h);
  }
  // one head partial per unit tile and epilogue warp slice of four warps
  p->head_slots = p->epi_warps / 4 * cdiv(h, kTcUnits);
  if (p->head_slots > tc_gate_tiles(h))
    IADMM_FAIL(IADMM_EMODE, "gate plan: %d head partials per row exceed the %d workspace slots", p->head_slots, tc_gate_tiles(h));
  return IADMM_OK;
}

static bool use_quads() {
  // 4-CTA multicast clusters are bit-identical to plain pairs but measured 3-4 % slower on B200 (the kernel is
  // bound by the per-SM request port, not by L2 reads, and only 132 SMs host 4-CTA clusters): development switch only.
  const char* e = dev_env("IADMM_TC_QUAD");
  return e && e[0] == '1';
}

static bool use_cta_pairs() {
  const char* e = dev_env("IADMM_TC_CTA_PAIR");      // development switch: 0 = single-CTA tiles
  return !(e && e[0] == '0');
}

int launch_gates_tc(const void* packed, const WeightLayout& L, const float* xv, const float* g, const __half* Hin_hi,
                    const __half* Hin_lo, __half* Hout_hi, __half* Hout_lo, float* H_out_f32, float* C,
                    float* head_part, long rows, int h, const GatePlan& plan, cudaStream_t st, float* gates_out, const TcIl* il) {
  const int nprod = plan.nprod;
  if (plan.interleaved != (il != nullptr)) IADMM_FAIL(IADMM_EMODE, "gate plan and row-interleaved state buffers disagree");
  if (h % 8 != 0) IADMM_FAIL(IADMM_EMODE, "tensor-core gate path needs hidden_dim %% 8 == 0");
  if (rows > 0x7fffffffL - 2 * kTcBM) IADMM_FAIL(IADMM_ESHAPE, "too many rows for one launch");
  int num_sms = 0, rc;
  if ((rc = device_sm_count(&num_sms))) return rc;
  if (const char* e = dev_env("IADMM_TC_MAX_SMS")) {      // development switch: restrict the persistent grid (this call only)
    const int v = atoi(e);
    if (v >= 2 && v < num_sms) num_sms = v;
  }
  const bool pair = use_cta_pairs() && num_sms >= 2;
  const char* base = static_cast<const char*>(packed);
  if (nprod == 2 && !pair) IADMM_FAIL(IADMM_EMODE, "the fp16+fp8 gate mode runs on CTA pairs only");
  if (nprod == 2 && h % 16 != 0 && !il) IADMM_FAIL(IADMM_EMODE, "the fp16+fp8 gate mode needs hidden_dim %% 16 == 0 outside the row-interleaved kernels");
  CUtensorMap ma_hi, ma_lo, mb_hi, mb_lo;
  const int b_box_rows = pair ? kPairBBoxRows : kTcBN;
  const int bk = pair ? kPairBK : kTcBK;
  int il_bk = 64;
  if (const char* e = dev_env("IADMM_TC_IL_BK")) il_bk = (atoi(e) == 32) ? 32 : 64;   // development switch
  if (il) {
    if (!pair || nprod != 2 || gates_out) IADMM_FAIL(IADMM_EMODE, "the row-interleaved layout is the F16F8 CTA-pair solve path only");
    if ((rc = get_map_il(&ma_hi, Hin_hi, (uint64_t)il->rows_p, h / 8, false, il_bk))) return rc;
    if ((rc = get_map_il(&ma_lo, Hin_lo, (uint64_t)il->rows_p, (h + 15) / 16, true, il_bk))) return rc;
    if ((rc = get_map_il(&mb_hi, base + L.off_uhi_il, (uint64_t)4 * h, h / 8, false, il_bk))) return rc;
    if ((rc = get_map_il(&mb_lo, base + L.off_uq8_il, (uint64_t)4 * h, (h + 15) / 16, true, il_bk))) return rc;
  } else {
    if ((rc = get_map(&ma_hi, Hin_hi, (uint64_t)rows, h, kTcBM, 2, bk))) return rc;
    if ((rc = get_map(&mb_hi, base + L.off_uhi, (uint64_t)4 * h, h, b_box_rows, 2, bk))) return rc;
    if (nprod == 2) {
      // packed e4m3 images: byte tensors [rows][q8_pitch], one 128-byte box row per 64-wide K block
      const int pitch = (int)q8_pitch(h);
      if ((rc = get_map(&ma_lo, Hin_lo, (uint64_t)rows, pitch, kTcBM, 1, 128))) return rc;
      if ((rc = get_map(&mb_lo, base + L.off_uq8, (uint64_t)4 * h, pitch, b_box_rows, 1, 128))) return rc;
    } else {
      if ((rc = get_map(&ma_lo, Hin_lo, (uint64_t)rows, h, kTcBM, 2, bk))) return rc;
      if ((rc = get_map(&mb_lo, base + L.off_ulo, (uint64_t)4 * h, h, b_box_rows, 2, bk))) return rc;
    }
  }

  TcParams P;
  P.wc = reinterpret_cast<const float*>(base + L.off_wc);
  P.bias = reinterpret_cast<const float*>(base + L.off_bias);
  P.wh = reinterpret_cast<const float*>(base + L.off_wh);
  P.scale = reinterpret_cast<const float*>(base + L.off_scale);
  P.tilep = reinterpret_cast<const float*>(base + (il ? L.off_tilep_il : L.off_tilep));
  P.xv = xv; P.g = g;
  P.hout_hi = Hout_hi; P.hout_lo = Hout_lo; P.hout_f32 = H_out_f32; P.C = C; P.head_part = head_part;
  P.gates_out = gates_out; P.exp = 0; P.wait_ns = IADMM_MBAR_SUSPEND_NS;
  P.rows_p = il ? il->rows_p : 0; P.c_rm_out = il ? il->C_rm_out : nullptr;
  if (il) P.C = il->C_il;
  P.rows = rows; P.h = h; P.q8_pitch = q8_pitch(h);
  P.unit_tiles = cdiv(h, kTcUnits);
  P.skew = 0;             // set at launch from the grid size (tile_unit)
  P.k_blocks = cdiv(h, il ? il_bk : bk);
  P.nprod = nprod;
  int exp_mode = 0, epi = 1;
  if (const char* e = dev_env("IADMM_TC_EXP")) exp_mode = atoi(e);          // development experiments, see TcParams::exp
  if (const char* w = dev_env("IADMM_TC_EPI")) {    // development switch: 0 = scalar epilogue, 1 = packed fp32 (default), 2 = packed + exp-only tanh
    epi = atoi(w);
    if (epi < 0 || epi > 3) epi = 1;                  // 3: shared-reciprocal activations (row-interleaved kernel only)
  }
  // IADMM_GATES_TC_F16F8U: the H-rounding correction product is not issued (TcParams::exp 7 is exactly that and numerically valid)
  if (plan.drop_h && exp_mode == 0) exp_mode = 7;
  const int epi_warps = plan.epi_warps;
  P.exp = exp_mode;
  if (const char* e = dev_env("IADMM_TC_WAIT_NS")) P.wait_ns = (uint32_t)atoi(e);
  // cluster size: 4 (two pairs sharing each U tile through TMA multicast) when there is enough work, else 2
  int cl = 1;
  if (pair) {
    cl = 2;
    const long row_tiles = (rows + 2 * kTcBM - 1) / (2 * kTcBM);
    if (use_quads() && row_tiles >= 2 && num_sms >= 4 && !gates_out && !il) cl = 4;
  }
  const int tile_rows = (pair ? 2 * kTcBM : kTcBM) * (cl == 4 ? 2 : 1);
  P.num_tiles = ((rows + tile_rows - 1) / tile_rows) * P.unit_tiles;
  const int a_bytes = pair ? kPairABytes : kTcABytes;
  const int b_bytes = pair ? kPairBBytes : kTcBBytes;
  const int stage_bytes = (nprod == 1) ? (a_bytes + b_bytes) : 2 * (a_bytes + b_bytes);
  P.stages = (192 * 1024) / stage_bytes;                 // 4 / 8 (single CTA, 32-wide K), 3 / 6 (pair, 64-wide K)
  if (il) P.stages = (192 * 1024) / (il_bk * 1024);      // 3 x 64 KB or 6 x 32 KB
  const size_t smem = 1024 + (size_t)P.stages * (il ? il_bk * 1024 : stage_bytes) + 2 * kParamFloats * sizeof(float) +
                      (2 * P.stages + 8) * sizeof(uint64_t) + 16;

  int threads = kTcThreads;
  if (pair) {
    auto launch = [&](auto kernel, PerDeviceOnce* attr_done, int cluster) -> int {
      int rc2;
      if ((rc2 = ensure_dyn_smem(kernel, 220 * 1024, attr_done))) return rc2;
      long clusters = num_sms / cluster;
      if (cluster == 4) {
        // co-resident 4-CTA clusters (GPC granularity: 33 on a 148-SM B200)
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3((unsigned)(num_sms / 4 * 4)); cfg.blockDim = dim3(kTcThreads); cfg.dynamicSmemBytes = smem;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = 4; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        int n = 0;
        if (cudaOccupancyMaxActiveClusters(&n, kernel, &cfg) != cudaSuccess || n <= 0) n = num_sms / 4 - 4;
        clusters = n < num_sms / 4 ? n : num_sms / 4;
      }
      if (P.num_tiles < clusters) clusters = P.num_tiles;
      P.skew = tile_skew_needed(clusters, P.unit_tiles, P.h);
      kernel<<<(unsigned)(cluster * clusters), threads, smem, st>>>(ma_hi, ma_lo, mb_hi, mb_lo, P);
      return IADMM_OK;
    };
    static PerDeviceOnce a34, a24, a14, a32, a22, a12, e0, e2, s2, s3, s1, i4, i5, i6, i7, i8;
    if (il && epi_warps == 16) {
      threads = pair_threads(7);
      // hidden_dim <= kEpi16MaxHidden: the special-function unit paces the epilogue (ncu: XU 47 % busy), and one shared reciprocal for the
      // four activations of a unit (4 ex2 + 1 rcp instead of 4 + 4) is 10 % faster (0.649 -> 0.586 ms at hidden_dim 208,
      // profiles/r02_gate_shared_rcp_ab.jsonl); in the power-capped 8-warp regime the same change is 1 % SLOWER (more ALU
      // instructions), so it stays a development switch there.  IADMM_TC_EPI=1 forces the separate reciprocals here.
      static PerDeviceOnce i9, i10;
      if (dev_env("IADMM_TC_EPI") && epi == 1)      rc = launch(gates_tc_pair_kernel<2, 2, 7>, &i7, 2);
      else if (dev_env("IADMM_TC_EPI") && epi == 2) rc = launch(gates_tc_pair_kernel<2, 2, 10>, &i10, 2);
      else                                          rc = launch(gates_tc_pair_kernel<2, 2, 9>, &i9, 2);
    } else if (il) {
      if (epi == 3)         rc = launch(gates_tc_pair_kernel<2, 2, 8>, &i8, 2);
      else if (epi == 2)    rc = launch(gates_tc_pair_kernel<2, 2, 6>, &i6, 2);
      else if (il_bk == 32) rc = launch(gates_tc_pair_kernel<2, 2, 5>, &i5, 2);
      else                  rc = launch(gates_tc_pair_kernel<2, 2, 4>, &i4, 2);
    } else if (gates_out) {        // training forward: the epilogue also stores the gate activations
      if (nprod == 1)      rc = launch(gates_tc_pair_kernel<1, 2, 0>, &s1, 2);
      else if (nprod == 3) rc = launch(gates_tc_pair_kernel<3, 2, 3>, &s3, 2);
      else                 rc = launch(gates_tc_pair_kernel<2, 2, 3>, &s2, 2);
    } else if (cl == 4) {
      if (nprod == 3)      rc = launch(gates_tc_pair_kernel<3, 4, 1>, &a34, 4);
      else if (nprod == 2) rc = launch(gates_tc_pair_kernel<2, 4, 1>, &a24, 4);
      else                 rc = launch(gates_tc_pair_kernel<1, 4, 1>, &a14, 4);
    } else {
      if (nprod == 3)      rc = launch(gates_tc_pair_kernel<3, 2, 1>, &a32, 2);
      else if (nprod == 2 && epi == 0) rc = launch(gates_tc_pair_kernel<2, 2, 0>, &e0, 2);
      else if (nprod == 2 && epi == 2) rc = launch(gates_tc_pair_kernel<2, 2, 2>, &e2, 2);
      else if (nprod == 2) rc = launch(gates_tc_pair_kernel<2, 2, 1>, &a22, 2);
      else                 rc = launch(gates_tc_pair_kernel<1, 2, 1>, &a12, 2);
    }
    if (rc) return rc;
    IADMM_LAUNCH_CHECK("gates_tc_pair_kernel");
    return IADMM_OK;
  }
  const long grid = P.num_tiles < num_sms ? P.num_tiles : num_sms;
  P.skew = tile_skew_needed(grid, P.unit_tiles, P.h);
  static PerDeviceOnce a3, a1;
  if (nprod == 3) {
    if ((rc = ensure_dyn_smem(gates_tc_kernel<3>, 220 * 1024, &a3))) return rc;
    gates_tc_kernel<3><<<(unsigned)grid, kTcThreads, smem, st>>>(ma_hi, ma_lo, mb_hi, mb_lo, P);
  } else {
    if ((rc = ensure_dyn_smem(gates_tc_kernel<1>, 220 * 1024, &a1))) return rc;
    gates_tc_kernel<1><<<(unsigned)grid, kTcThreads, smem, st>>>(ma_hi, ma_lo, mb_hi, mb_lo, P);
  }
  IADMM_LAUNCH_CHECK("gates_tc_kernel");
  return IADMM_OK;
}

}  // namespace iadmm

// Shared device helpers and the internal (non-ABI) kernel launch interface of libiadmm_b200.
// sm_100a only.  Nothing here is visible through include/iadmm.h.
#pragma once

#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stddef.h>

#include "../../include/iadmm.h"

namespace iadmm {

// ------------------------------------------------------------------------------------------------
// error plumbing (thread-local last-error string, set by IADMM_FAIL / IADMM_CUDA)
// ------------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);

#define IADMM_FAIL(code, ...)                      \
  do {                                             \
    ::iadmm::set_error(__VA_ARGS__);               \
    return (code);                                 \
  } while (0)

#define IADMM_CUDA(expr)                                                                       \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) {                                                                   \
      ::iadmm::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return IADMM_ECUDA;                                                                      \
    }                                                                                          \
  } while (0)

#define IADMM_LAUNCH_CHECK(name)                                                               \
  do {                                                                                         \
    cudaError_t _e = cudaGetLastError();                                                       \
    if (_e != cudaSuccess) {                                                                   \
      ::iadmm::set_error("launch of %s failed: %s", name, cudaGetErrorString(_e));             \
      return IADMM_ECUDA;                                                                      \
    }                                                                                          \
  } while (0)

// ------------------------------------------------------------------------------------------------
// per-device facts and opt-ins.  cudaFuncSetAttribute and the SM count are per DEVICE: a process that drives several GPUs
// (the Python layer wraps every call in torch.cuda.device(dev)) needs the opt-in on each of them, so the "already done"
// marks are bit masks over the device ordinal, never plain process-wide flags.
// ------------------------------------------------------------------------------------------------
constexpr int kMaxDevices = 64;
struct PerDeviceOnce { unsigned long long done = 0ull; };     // bit d: attribute set on device d (benign if set twice)
int device_sm_count(int* sms);                                // SM count of the CURRENT device (cached per ordinal)
int check_device();                                           // IADMM_EARCH unless the CURRENT device is sm_100

template <typename KernelT>
static inline int ensure_dyn_smem(KernelT kernel, int bytes, PerDeviceOnce* once) {
  int dev = 0;
  IADMM_CUDA(cudaGetDevice(&dev));
  const unsigned long long bit = (dev >= 0 && dev < kMaxDevices) ? (1ull << dev) : 0ull;
  if (bit && (__atomic_load_n(&once->done, __ATOMIC_ACQUIRE) & bit)) return IADMM_OK;
  IADMM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  if (bit) __atomic_fetch_or(&once->done, bit, __ATOMIC_RELEASE);
  return IADMM_OK;
}

// Development switches (IADMM_TC_*, IADMM_RESIDENT, ...) are read from the environment ONLY in a development build
// (`IADMM_DEV_BUILD=1 python i-admm-lstm_b200/build.py` -> libiadmm_b200_dev.so, compiled with -DIADMM_DEV_SWITCHES).
// The release library never calls getenv: no environment variable can change what it computes.
const char* dev_env(const char* name);

// measurement spans (iadmm_profile_begin/_end, include/iadmm.h): no-ops unless a profile is open
enum { kProfKkt = 0, kProfGates = 1, kProfTail = 2,            // iadmm_solve: KKT passes+combines | gate kernel | tail
       kProfTrainGates = 3,                                     // training forward: gate kernel (+ state split)
       kProfTrainGemm = 4,                                      // training backward: the two gate-product adjoint GEMMs (+ operand splits)
       kProfTrainKkt = 5,                                       // training: KKT passes of forward, residuals and adjoint
       kProfTrainCell = 6,                                      // training backward: cell adjoint + small parameter adjoints
       kProfKinds = 7 };
void prof_begin(int kind, cudaStream_t st);
void prof_end(int kind, cudaStream_t st);

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
static inline int    cdiv(int a, int b) { return (a + b - 1) / b; }
static inline bool   aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ------------------------------------------------------------------------------------------------
// packed weights (layout computed on the host from (h, length); see pack.cu)
// ------------------------------------------------------------------------------------------------
constexpr int   kHShift = 14;   // H is stored as fp16 hi/lo of H * 2^14 (|H| < 1 for an LSTM state)
constexpr int   kSchedStride = 6;   // floats per schedule row, see Sched below

struct WeightLayout {
  int    h, length;
  size_t off_u32;     // fp32 [h][4h]   column 4*j+g  (g: 0=i 1=f 2=o 3=u)
  size_t off_wc;      // fp32 [2][4h]   W rows, same column order
  size_t off_bias;    // fp32 [4h]
  size_t off_wh;      // fp32 [h]
  size_t off_bh;      // fp32 [1] (+pad)
  size_t off_sched;   // fp32 [length][6]: rho_ineq, rho_eq, 1/rho_ineq, 1/rho_eq, alpha, 1-alpha
  size_t off_scale;   // fp32 [4]: u_scale (power of two applied to U before the fp16 split),
                      //           dequant = 1/(u_scale*2^14), |U|max, unused
  size_t off_uhi;     // fp16 [4h][h]   row 4*j+g, K-major (k = input unit): tcgen05 B operand, hi part
  size_t off_ulo;     // fp16 [4h][h]   lo part
  size_t off_u32hi;   // fp16 [h][4h]   hi part of U*2^s in the fp32 image's layout (K-major for H_bar = D U^T)
  size_t off_u32lo;   // fp16 [h][4h]   lo part
  size_t off_uq8;     // e4m3 [4h][q8_pitch(h)]: per 64-wide K block 64 B of residual (U*2^s - fp16(U*2^s)) * 2^6 followed by
                      //                64 B of the coarse copy fp16(U*2^s) * 2^-5   (F16F8 mode; one 128-byte TMA row)
  size_t off_tilep;   // fp32 [ceil(h/64)][832]: per 64-unit tile the W row 0 | W row 1 | bias (256 gate columns each) | W_h (64) block the
                      //                gate kernel's epilogue reads, contiguous so ONE bulk copy stages it in shared memory
  size_t off_tilep_il;// the same blocks with the gate columns in the order of the row-interleaved kernels (il_gate_col)
  size_t off_uhi_il;  // fp16 [h/8][4h][8]: row-interleaved image of fp16(U*2^s) (16-byte K groups of consecutive gate columns adjacent;
                      //                the no-swizzle UMMA core-matrix order, see gates_tc.cu "row-interleaved layout")
  size_t off_uq8_il;  // e4m3 [ceil(h/16)][2][4h][16]: residual plane, coarse plane per 16-wide K group
  size_t total;
};
// Gate-column order of the row-interleaved gate kernels.  Everywhere else column c = 4 * unit + gate (i, f, o, u).  The
// row-interleaved U images and parameter blocks keep, within every 8 columns (two hidden units), the same gate of the two
// units adjacent: (i0 i1 f0 f1 o0 o1 u0 u1).  The accumulator columns a thread reads from tensor memory are then already the
// operand pairs of the epilogue's two-wide fp32 instructions (one pair = one gate of two units), for every activation and the
// state update alike, instead of (i, f) / (o, u) pairs of one unit that have to be re-paired by register moves.
__host__ __device__ __forceinline__ int il_gate_col(int c)     { return (c & ~7) | ((c & 3) << 1) | ((c >> 2) & 1); }
__host__ __device__ __forceinline__ int il_gate_col_inv(int q) { return (q & ~7) | ((q & 1) << 2) | ((q >> 1) & 3); }
WeightLayout weight_layout(int h, int length);

struct Sched {  // one schedule row, already in fp32 exactly as models/lstm.py:60-63 rounds it
  float rho_ineq, rho_eq, inv_rho_ineq, inv_rho_eq, alpha, one_minus_alpha;
};

// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------
#ifdef __CUDACC__

constexpr unsigned kFullMask = 0xffffffffu;

// sm_100 two-wide fp32 arithmetic (FFMA2 / FMUL2 / FADD2): each lane of a pair is the same IEEE operation as the scalar
// instruction, at half the issue slots.  NOTE: ptxas contracts mul.f32x2 + add.f32x2 into FFMA2 even with .rn, so keep
// products that the reference rounds separately in scalar __fmul_rn/__fadd_rn form.
typedef unsigned long long u64;
__device__ __forceinline__ u64 pk2(float a, float b) { u64 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ u64 bc2(float a) { u64 r; asm("mov.b64 %0, {%1, %1};" : "=l"(r) : "f"(a)); return r; }
__device__ __forceinline__ void upk2(u64 v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) { u64 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ u64 mul2(u64 a, u64 b) { u64 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 add2(u64 a, u64 b) { u64 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }

// streaming 128-bit load: read-only path, do not allocate in L1 (matrix data is touched once per pass)
__device__ __forceinline__ float4 ldg_stream4(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
// same, through the coherent path (for buffers that are rewritten in place by the same kernel)
__device__ __forceinline__ float4 ld_stream4_coherent(const float* p) {
  float4 r;
  asm volatile("ld.global.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ float ldg_stream1(const float* p) {
  float r;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
  return r;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(kFullMask, v, o));
  return v;
}

// Transpose-reduce: every lane holds NV partial values; afterwards lane l holds the warp-wide total of
// value (l * NV) >> 5  (i.e. 32/NV consecutive lanes hold the same value index).  NV in {1,2,4,8,16,32}.
// NV shuffles + log2(32/NV) more instead of 5*NV.  Fixed order => deterministic.
template <int NV, bool IS_MAX = false>
__device__ __forceinline__ float warp_transpose_reduce(float (&v)[NV], int lane) {
  int bit = 16;
#pragma unroll
  for (int half = NV / 2; half >= 1; half >>= 1) {
    const bool upper = (lane & bit) != 0;
#pragma unroll
    for (int i = 0; i < half; ++i) {
      const float send = upper ? v[i] : v[i + half];
      const float keep = upper ? v[i + half] : v[i];
      const float got  = __shfl_xor_sync(kFullMask, send, bit);
      v[i] = IS_MAX ? fmaxf(keep, got) : keep + got;
    }
    bit >>= 1;
  }
  float r = v[0];
#pragma unroll
  for (; bit >= 1; bit >>= 1) {
    const float got = __shfl_xor_sync(kFullMask, r, bit);
    r = IS_MAX ? fmaxf(r, got) : r + got;
  }
  return r;
}

// 1/(1+exp(-x)) the way torch's CUDA sigmoid evaluates it (fp32 expf, IEEE divide)
__device__ __forceinline__ float sigmoid_ref(float x) { return 1.0f / (1.0f + expf(-x)); }

#endif  // __CUDACC__

// ------------------------------------------------------------------------------------------------
// internal launchers (each enqueues on `st`; returns IADMM_OK or an error code with message set)
// ------------------------------------------------------------------------------------------------
struct KktDims {
  int B, n, m, num_ineq;
  int rows_per_chunk;          // R: rows of Q / A0 one CTA streams (multiple of 8)
  int chunks_q, chunks_a;      // ceil(n/R), ceil(m/R)
  int sum_q, sum_a;            // column partials the combine kernels add up (1 once folded into chunk 0, else = chunks)
};
KktDims make_kkt_dims(int B, int n, int m, int num_ineq);
int kkt_sum_chunks(int chunks);   // partials left to add after launch_kkt_combine1/2 (1 when they were folded)
KktDims make_kkt_dims_train(int B, int n, int m, int num_ineq);   // batch-aware chunking for the training entry points

struct KktScratch {            // all [B, ...] fp32, carved from the solve workspace
  float* qxt;   // [B,n]   Q  x~          (pass 1)
  float* qx;    // [B,n]   Q  x           (pass 1, residual of the previous iterate)
  float* axt;   // [B,m]   A0 x~
  float* ax;    // [B,m]   A0 x
  float* aw1;   // [B,m]   A0 w1          (pass 2)
  float* part_a;  // [B, chunks_a, 2, n]  column partials of A0^T {v | y} (pass 1) / A0^T w2 (pass 2, slot 0)
  float* part_q;  // [B, chunks_q, n]     column partials of Q^T w1     (pass 2)
  float* w;     // [B, n+m]  K xv - rhs
  float* g;     // [B, n+m]  K^T w
  float *x_old, *y_old, *z_old;   // [B,n], [B,m], [B,m]: the iterate BEFORE the last tail update (linear-system residual trace)
};
constexpr int kMetricRows = 6;   // rows of one metric_trace block: objective, ineq max/mean, eq max/mean, ||K xv - rhs||
size_t kkt_scratch_floats(const KktDims& d);
void   kkt_scratch_carve(const KktDims& d, float* base, KktScratch* s);

// A matrix batch in "bitmap slab" sparse form (sparse.cu; layout documented at iadmm_sparse_pack in include/iadmm.h)
struct SpMat {
  const uint4*    mask;        // [B][rows][S] 128-bit occupancy masks
  const uint32_t* off;         // [B][rows][S] offset of the slab's first value inside the instance's values
  const float*    vals;        // [B][cap]     non-zero values, row-major per instance; NULL = matrix not given in sparse form
  int    S;                    // slabs per row = ceil(n / 128)
  size_t mask_stride;          // rows * S   (entries per instance of mask and off)
  size_t vals_stride;          // cap
  // -- or: the dense matrix with block skipping (vals == NULL): one bit per 8-row x 128-column block
  const unsigned long long* blk;   // [B][ceil(rows/8)] bit s of word g: block (g, s) holds a non-zero; NULL = not given
  size_t blk_stride;               // ceil(rows/8)
};
struct KktSparse { SpMat q, a; };
int sparse_view(const void* packed, int B, int rows, int n, size_t cap, SpMat* out);   // carve a packed buffer

// Programmatic dependent launch (PDL) inside one iteration of the solve: a kernel launched with `pdl` may become resident while
// the kernel before it in the stream drains (that kernel executes `pdl_trigger()` first thing), runs its prologue, and blocks in
// `pdl_wait()` until the predecessor has completed and its writes are visible -- BEFORE its first read of anything a predecessor
// wrote and before its first global write.  Kernels carry both instructions unconditionally (no-ops in a normal launch).
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
template <typename... KArgs, typename... Args>
static inline void launch_kernel_pdl(bool pdl, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                     Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = pdl ? 1 : 0;
  cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#endif

// pass 1: qxt,qx,axt,ax and column partials of A0^T v, A0^T y.  `pdl`: see above; only valid when NOTHING the pass reads
// (incl. Q and A0, which its copy-engine producer streams without waiting) was written by the kernel before it in the stream.
int launch_kkt_pass1(const KktDims& d, const float* Q, const float* A0, const float* xv, const float* x,
                     const float* y, const KktScratch& s, cudaStream_t st, const KktSparse* sp = nullptr, bool pdl = false);
// combine 1: w = K xv - rhs ; residual norms of (x,y,z) into trace row `trace_row` (skipped when < 0)
int launch_kkt_combine1(const KktDims& d, const float* p, const float* xv, const float* x, const float* y,
                        const float* z, const Sched* sched_t, float sigma, const KktScratch& s,
                        float* pri_trace, float* dual_trace, float* pri_trace_u, float* dual_trace_u,
                        const float* sd, const float* se, const float* sc, int trace_row, int residual_only,
                        cudaStream_t st, float* metric_trace = nullptr, const float* zu = nullptr,
                        const Sched* sched_prev = nullptr, bool pdl = false);
// pass 2: column partials of Q^T w1, A0^T w2 and rows A0 w1
int launch_kkt_pass2(const KktDims& d, const float* Q, const float* A0, const KktScratch& s, cudaStream_t st,
                     const KktSparse* sp = nullptr, bool pdl = false);
// combine 2: g = K^T w
int launch_kkt_combine2(const KktDims& d, const Sched* sched_t, float sigma, const KktScratch& s, cudaStream_t st, bool pdl = false);

// LSTM cell on every coordinate (fp32 SIMT path): reads H_in, writes H_out, updates C in place,
// writes per-unit-tile partial sums of the output head into head_part [tiles][rows].
int  simt_gate_tiles(int h);
int  launch_gates_simt(const void* packed, const WeightLayout& L, const float* xv, const float* g,
                       const float* H_in, float* H_out, float* C, float* head_part, long rows, int h,
                       cudaStream_t st, float* gates_out = nullptr);

// tensor-core path (gate_tc.cu)
struct TcState {               // fp16 hi/lo images of H * 2^14, ping-pong.  In F16F8 mode the `lo` buffer holds the packed
  __half* h_hi[2];             // e4m3 image instead: [rows][q8_pitch(h)] bytes, per 64-wide K block 64 B of residual*2^5
  __half* h_lo[2];             // followed by 64 B of the coarse copy (H*2^14)*2^-6 (one 128-byte TMA row per block)
};
// bytes per row of a packed e4m3 operand pair
static inline size_t q8_pitch(int h) { return (size_t)((h + 63) / 64) * 128; }
// F16F8 scalings (powers of two, exact): residual of H*2^14 is < 4 -> *2^5 < 128; H*2^14*2^-6 < 256;
// fp16(U*2^s) < 2^13 -> *2^-5 < 256; residual of U*2^s is < 2 -> *2^6 < 128  (e4m3 max = 448)
constexpr int kQ8HLoShift = 5, kQ8HHiShift = -6, kQ8UHiShift = -5, kQ8ULoShift = 6;
int  tc_gate_tiles(int h);                    // head-partial slots to allocate
size_t tc_state_bytes(long rows, int h);
// Row-interleaved state layout of the fused solve (F16F8 mode): every per-row array is stored [column group][row][16 or 32 B]
// so that the thread-per-row epilogue reads and writes whole 128-byte lines (see gates_tc.cu).  rows_p = rows rounded up to 128.
struct TcIl {
  long   rows_p;
  float* C_il;        // fp32 [h/8][rows_p][8], the cell state between iterations
  float* C_rm_out;    // non-NULL on the last iteration: also write the caller's row-major C [rows][h]
};
static inline long il_rows(long rows) { return (rows + 127) / 128 * 128; }
// bytes of one row-interleaved e4m3 plane pair [ceil(h/16)][residual | coarse][rows_p][16]; with hidden_dim % 16 == 8 the last
// 16-unit group is half padding, which must read as zero (it is multiplied)
static inline size_t il_q8_bytes(long rows_p, int h) { return (size_t)((h + 15) / 16) * 2 * (size_t)rows_p * 16; }

// The gate-contraction path of one call: which kernels run, with how many products, and how many head partials per row the
// tail has to sum.  plan_gates (gates_tc.cu) is the one place that decides it; no caller compares against IADMM_GATES_*.
enum { kGatesFp32 = 0, kGatesResident = 1, kGatesTc = 2 };
struct GatePlan {
  int  path;          // kGatesFp32: CUDA cores; kGatesResident: on-chip-resident solve (resident.cu); kGatesTc: streaming tensor cores
  int  nprod;         // tensor-core products: 1 (fp16), 2 (fp16 + e4m3 corrections) or 3 (fp16 hi/lo split); 0 on CUDA cores
  bool interleaved;   // the solve keeps its state row-interleaved between iterations (TcIl)
  bool drop_h;        // IADMM_GATES_TC_F16F8U on the row-interleaved kernels: the e4m3 product that corrects the fp16 rounding
                      // of H is not issued
  int  epi_warps;     // epilogue warps of the tensor-core gate kernel (8 or 16)
  int  head_slots;    // head partials per row the gate kernel writes = what the tail sums (0 on the resident path)
};
// `training`: the forward of iadmm_step_fwd / iadmm_train_window, which never runs resident or row-interleaved (K and flags
// are then ignored).  Returns IADMM_EMODE, message set, for every mode / shape / flag combination no path serves.
int  plan_gates(int mode, int h, int n, int m, int K, int flags, bool training, GatePlan* plan);

int  launch_gates_tc(const void* packed, const WeightLayout& L, const float* xv, const float* g,
                     const __half* Hin_hi, const __half* Hin_lo, __half* Hout_hi, __half* Hout_lo,
                     float* H_out_f32 /* may be NULL */, float* C, float* head_part, long rows, int h,
                     const GatePlan& plan, cudaStream_t st, float* gates_out = nullptr, const TcIl* il = nullptr);
int  launch_split_state_il(const float* H, __half* hi, __half* q8, long rows, int h, cudaStream_t st);
int  launch_c_to_il(const float* C, float* C_il, long rows, int h, cudaStream_t st);
int  launch_split_state(const float* H, __half* hi, __half* lo, long rows, int h, int nprod, cudaStream_t st);
int  launch_zero_state(__half* hi, __half* lo, long rows, int h, int nprod, cudaStream_t st);
size_t tc_lo_bytes(long rows, int h);   // size of one `lo` buffer (fits both the fp16 and the packed e4m3 form)

// O(N) tail: xv -= head ; x,z,y updates (models/lstm.py:82-94)
// on-chip-resident solve for small instances (resident.cu): whether the shape fits it
bool resident_eligible(int n, int m, int h, int nprod);
int launch_solve_resident(const void* packed, const WeightLayout& L, const float* Q, const float* p, const float* A0,
                          const float* zl, const float* zu, const float* sd, const float* se, const float* sc, float* x, float* y,
                          float* z, float* xv, float* H, float* C, float* pri, float* dual, float* pri_u, float* dual_u,
                          float* metrics, int B, int n, int m, int num_ineq, int t0, int K, float sigma, int nprod, int flags,
                          cudaStream_t st);
int launch_tail(const KktDims& d, const float* head_part, int tiles, const float* b_h, const Sched* sched_t,
                const float* zl, const float* zu, float* x, float* y, float* z, float* xv, cudaStream_t st,
                const KktScratch* keep_old = nullptr);

}  // namespace iadmm

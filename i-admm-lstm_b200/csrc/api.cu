// extern "C" entry points of libiadmm_b200.so (declared in include/iadmm.h) and the per-iteration
// orchestration of the unrolled solve (main.py:874-887 x models/lstm.py:47-96 x utils.py:68-71).
#include "common.cuh"

#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

namespace iadmm {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

const char* dev_env(const char* name) {
#ifdef IADMM_DEV_SWITCHES
  return getenv(name);
#else
  (void)name;
  return nullptr;
#endif
}

int device_sm_count(int* sms) {
  static int cache[kMaxDevices] = {0};
  int dev = 0;
  IADMM_CUDA(cudaGetDevice(&dev));
  int v = (dev >= 0 && dev < kMaxDevices) ? __atomic_load_n(&cache[dev], __ATOMIC_RELAXED) : 0;
  if (!v) {
    IADMM_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev));
    if (dev >= 0 && dev < kMaxDevices) __atomic_store_n(&cache[dev], v, __ATOMIC_RELAXED);
  }
  *sms = v;
  return IADMM_OK;
}

// implemented in the other translation units
int pack_weights_impl(const float* const W[4], const float* const U[4], const float* const b[4], const float* W_h,
                      const float* b_h, const float* rho, const float* alpha, int h, int length, void* packed,
                      cudaStream_t st);
size_t ruiz_ws_floats(int B, int n, int m, int* R_out, int* cq_out, int* ca_out);
int ruiz_impl(const float* Q, const float* p, const float* A0, const float* zl, const float* zu, float* Qs, float* ps,
              float* A0s, float* zls, float* zus, float* d, float* e, float* c, int B, int n, int m, int iterations,
              void* workspace, size_t workspace_bytes, cudaStream_t st);
int launch_kkt_pass1_plain(const KktDims& d, const float* Q, const float* A0, const float* x, const float* y,
                           const KktScratch& s, cudaStream_t st);
int launch_kkt_penalty_diag(int B, int n, int m, int num_ineq, const Sched* sched_t, float* K, cudaStream_t st);
int launch_build_kkt(int B, int n, int m, int num_ineq, const float* Q, const float* p, const float* A0,
                     const float* x, const float* y, const float* z, const Sched* sched_t, float sigma, float* K,
                     float* rhs, float* rho_vec, cudaStream_t st);

int check_device() {
  int dev = 0, major = 0;
  IADMM_CUDA(cudaGetDevice(&dev));
  IADMM_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  if (major != 10) IADMM_FAIL(IADMM_EARCH, "device %d has compute capability %d.x; libiadmm_b200 needs sm_100 (B200)", dev, major);
  return IADMM_OK;
}

struct SolveWs {
  KktDims d;
  KktScratch s;
  float* head_part;       // [tiles][rows]
  float* h_alt;           // SIMT: second fp32 H buffer [rows,h]
  TcState tc;             // TC: fp16 hi/lo ping-pong
  float* c_il;            // F16F8: row-interleaved cell state [h/8][rows_p][8] (see gates_tc.cu)
  long rows_p;
  size_t bytes;
};

// measurement hooks: CUDA-event spans recorded around the phases of each iteration (bench.py)
struct ProfSpan { int kind; cudaEvent_t e0, e1; };
struct Profile {
  bool on = false;
  int cap = 0, used = 0;            // spans
  ProfSpan* span = nullptr;
  int open[kProfKinds];             // index of the span opened last per kind, -1 = none
};
static Profile g_prof;

void prof_begin(int kind, cudaStream_t st) {
  if (!g_prof.on || g_prof.used >= g_prof.cap) return;
  const int i = g_prof.used++;
  g_prof.span[i].kind = kind;
  g_prof.open[kind] = i;
  cudaEventRecord(g_prof.span[i].e0, st);
}
void prof_end(int kind, cudaStream_t st) {
  if (!g_prof.on || g_prof.open[kind] < 0) return;
  cudaEventRecord(g_prof.span[g_prof.open[kind]].e1, st);
  g_prof.open[kind] = -(g_prof.open[kind] + 2);       // closed: remembered as -(i+2)
}

// The layout depends on the gate mode alone (the path and the product count of the plan), not on K or the flags: one
// workspace serves every call of a mode, and resumed calls find the planes where the previous call left them.
static void plan_workspace(int B, int n, int m, int num_ineq, int h, const GatePlan& gp, void* base, SolveWs* ws) {
  const bool tc = gp.path != kGatesFp32;
  ws->d = make_kkt_dims(B, n, m, num_ineq);
  const size_t rows = (size_t)B * (n + m);
  const int tiles = tc ? tc_gate_tiles(h) : simt_gate_tiles(h);       // bound of the plan's head_slots
  char* p = static_cast<char*>(base);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 1024); return base ? p + o : nullptr; };
  float* kkt = reinterpret_cast<float*>(take(kkt_scratch_floats(ws->d) * sizeof(float)));
  if (base) kkt_scratch_carve(ws->d, kkt, &ws->s);
  ws->head_part = reinterpret_cast<float*>(take((size_t)tiles * rows * sizeof(float)));
  ws->h_alt = nullptr; ws->c_il = nullptr; ws->rows_p = (long)rows;
  memset(&ws->tc, 0, sizeof(ws->tc));
  if (tc) {
    // the F16F8 solve keeps its state row-interleaved: rows padded to a multiple of 128
    const bool il = gp.nprod == 2;
    ws->rows_p = il ? il_rows((long)rows) : (long)rows;
    const size_t rp = (size_t)ws->rows_p;
    const size_t hb = rp * (size_t)h * sizeof(__half);
    const size_t qb = il_q8_bytes((long)rp, h);                     // row-interleaved e4m3 planes [ceil(h/16)][2][rows_p][16]
    size_t lb = tc_lo_bytes((long)rows, h);
    if (il && hb > lb) lb = hb;
    if (il && qb > lb) lb = qb;
    for (int i = 0; i < 2; ++i) {
      ws->tc.h_hi[i] = reinterpret_cast<__half*>(take(hb));
      ws->tc.h_lo[i] = reinterpret_cast<__half*>(take(lb));
    }
    ws->c_il = il ? reinterpret_cast<float*>(take(rp * (size_t)h * sizeof(float))) : nullptr;
  } else {
    ws->h_alt = reinterpret_cast<float*>(take(rows * (size_t)h * sizeof(float)));
  }
  ws->bytes = off;
}

}  // namespace iadmm

using namespace iadmm;

extern "C" {

int iadmm_abi_version(void) { return IADMM_ABI_VERSION; }
const char* iadmm_last_error(void) { return g_err; }
int iadmm_device_check(void) { return check_device(); }

int iadmm_weights_bytes(int h, int length, size_t* bytes) {
  if (h <= 0 || length <= 0 || !bytes) IADMM_FAIL(IADMM_ESHAPE, "weights_bytes: h=%d length=%d", h, length);
  *bytes = weight_layout(h, length).total;
  return IADMM_OK;
}

int iadmm_pack_weights(const float* W_i, const float* U_i, const float* b_i, const float* W_f, const float* U_f,
                       const float* b_f, const float* W_o, const float* U_o, const float* b_o, const float* W_u,
                       const float* U_u, const float* b_u, const float* W_h, const float* b_h, const float* rho,
                       const float* alpha, int h, int length, void* packed, void* stream) {
  if (h <= 0 || length <= 0) IADMM_FAIL(IADMM_ESHAPE, "pack_weights: h=%d length=%d", h, length);
  const float* W[4] = {W_i, W_f, W_o, W_u};
  const float* U[4] = {U_i, U_f, U_o, U_u};
  const float* b[4] = {b_i, b_f, b_o, b_u};
  for (int g = 0; g < 4; ++g)
    if (!W[g] || !U[g] || !b[g]) IADMM_FAIL(IADMM_EALIGN, "pack_weights: NULL gate parameter %d", g);
  if (!W_h || !b_h || !rho || !alpha || !packed) IADMM_FAIL(IADMM_EALIGN, "pack_weights: NULL pointer");
  if (!aligned16(packed)) IADMM_FAIL(IADMM_EALIGN, "pack_weights: packed buffer not 16-byte aligned");
  int rc = check_device();
  if (rc) return rc;
  return pack_weights_impl(W, U, b, W_h, b_h, rho, alpha, h, length, packed, static_cast<cudaStream_t>(stream));
}

int iadmm_ruiz_workspace_bytes(int B, int n, int m, size_t* bytes) {
  if (B <= 0 || n <= 0 || m < 0 || !bytes) IADMM_FAIL(IADMM_ESHAPE, "ruiz_workspace_bytes: B=%d n=%d m=%d", B, n, m);
  *bytes = ruiz_ws_floats(B, n, m, nullptr, nullptr, nullptr) * sizeof(float);
  return IADMM_OK;
}

int iadmm_ruiz(const float* Q, const float* p, const float* A0, const float* zl, const float* zu, float* Qs, float* ps,
               float* A0s, float* zls, float* zus, float* d, float* e, float* c, int B, int n, int m, int iterations,
               void* workspace, size_t workspace_bytes, void* stream) {
  if (B <= 0 || n <= 0 || m < 0 || iterations < 0) IADMM_FAIL(IADMM_ESHAPE, "ruiz: B=%d n=%d m=%d ites=%d", B, n, m, iterations);
  if (B > 65535) IADMM_FAIL(IADMM_ESHAPE, "ruiz: batch %d > 65535 per call", B);
  if (!Q || !p || !Qs || !ps || !d || !c || !workspace) IADMM_FAIL(IADMM_EALIGN, "ruiz: NULL pointer");
  if (m > 0 && (!A0 || !zl || !zu || !A0s || !zls || !zus || !e)) IADMM_FAIL(IADMM_EALIGN, "ruiz: NULL constraint pointer");
  if (Q == Qs || (m > 0 && A0 == A0s)) IADMM_FAIL(IADMM_EALIGN, "ruiz: outputs must not alias inputs");
  int rc = check_device();
  if (rc) return rc;
  return ruiz_impl(Q, p, A0, zl, zu, Qs, ps, A0s, zls, zus, d, e, c, B, n, m, iterations, workspace, workspace_bytes,
                   static_cast<cudaStream_t>(stream));
}

int iadmm_solve_workspace_bytes(int B, int n, int m, int h, int mode, size_t* bytes) {
  if (B <= 0 || n <= 0 || m < 0 || h <= 0 || !bytes) IADMM_FAIL(IADMM_ESHAPE, "solve_workspace_bytes: B=%d n=%d m=%d h=%d", B, n, m, h);
  GatePlan gp;
  int rc = plan_gates(mode, h, n, m, 1, 0, false, &gp);
  if (rc) return rc;
  SolveWs ws;
  plan_workspace(B, n, m, 0, h, gp, nullptr, &ws);
  *bytes = ws.bytes;
  return IADMM_OK;
}

static int solve_impl(const void* packed_weights, const float* Q, const float* p, const float* A0, const float* zl,
                const float* zu, const float* sd, const float* se, const float* sc, float* x, float* y, float* z,
                float* xv, float* H, float* C, float* pri_trace, float* dual_trace, float* pri_trace_u,
                float* dual_trace_u, float* metric_trace, int B, int n, int num_ineq, int num_eq, int h, int length, int t0, int K,
                float sigma, int mode, int flags, void* workspace, size_t workspace_bytes, void* stream, const KktSparse* sp) {
  const int m = num_ineq + num_eq;
  const bool spq = sp && sp->q.vals, spa = sp && sp->a.vals;     // bitmap-slab form: the dense pointer is not needed
  if (B <= 0 || n <= 0 || num_ineq < 0 || num_eq < 0 || h <= 0 || K < 0 || t0 < 0)
    IADMM_FAIL(IADMM_ESHAPE, "solve: B=%d n=%d ineq=%d eq=%d h=%d t0=%d K=%d", B, n, num_ineq, num_eq, h, t0, K);
  if (t0 + K > length) IADMM_FAIL(IADMM_ESHAPE, "solve: iterations %d..%d exceed the schedule length %d (lstm.py:60)", t0, t0 + K - 1, length);
  if (B > 65535) IADMM_FAIL(IADMM_ESHAPE, "solve: batch %d > 65535 per call; shard the batch", B);
  if (!packed_weights || (!Q && !spq) || !p || !x || !xv || !H || !C || !workspace) IADMM_FAIL(IADMM_EALIGN, "solve: NULL pointer");
  if (m > 0 && ((!A0 && !spa) || !zl || !zu || !y || !z)) IADMM_FAIL(IADMM_EALIGN, "solve: NULL constraint pointer");
  if ((pri_trace_u || dual_trace_u) && (!sd || !sc || (m > 0 && !se)))
    IADMM_FAIL(IADMM_EALIGN, "solve: un-scaled traces need the Ruiz diagonals d, e, c");
  if (!aligned16(H) || !aligned16(C) || !aligned16(workspace) || !aligned16(packed_weights))
    IADMM_FAIL(IADMM_EALIGN, "solve: H, C, workspace and packed weights must be 16-byte aligned");
  int rc = check_device();
  if (rc) return rc;
  GatePlan gp;
  if ((rc = plan_gates(mode, h, n, m, K, flags, false, &gp))) return rc;
  SolveWs ws;
  plan_workspace(B, n, m, num_ineq, h, gp, workspace, &ws);
  if (ws.bytes > workspace_bytes) IADMM_FAIL(IADMM_EWORK, "solve: workspace too small: %zu < %zu", workspace_bytes, ws.bytes);
  if (K == 0) return IADMM_OK;

  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const WeightLayout L = weight_layout(h, length);
  const char* wbase = static_cast<const char*>(packed_weights);
  const Sched* sched = reinterpret_cast<const Sched*>(wbase + L.off_sched);
  const float* b_h = reinterpret_cast<const float*>(wbase + L.off_bh);
  const long rows = (long)B * (n + m);
  const bool want_trace = pri_trace || dual_trace || pri_trace_u || dual_trace_u || metric_trace;

  if (gp.path == kGatesResident)
    return launch_solve_resident(packed_weights, L, Q, p, A0, zl, zu, sd, se, sc, x, y, z, xv, H, C, pri_trace, dual_trace,
                                 pri_trace_u, dual_trace_u, metric_trace, B, n, m, num_ineq, t0, K, sigma, gp.nprod, flags, st);

  float* hbuf[2] = {H, ws.h_alt};
  int cur = 0;
  const bool tc = gp.path == kGatesTc, il = gp.interleaved;
  // one iteration per call (main.py:874-887): the state stays in the planes the previous call left in this workspace
  const bool resume = (flags & IADMM_F_RESUME) != 0;
  if (resume && (flags & IADMM_F_ZERO_STATE)) IADMM_FAIL(IADMM_EMODE, "solve: IADMM_F_RESUME and IADMM_F_ZERO_STATE exclude each other");
  if (resume && (flags & IADMM_F_RESUME_ODD)) cur = 1;
  TcIl ilp;
  ilp.rows_p = ws.rows_p; ilp.C_il = ws.c_il; ilp.C_rm_out = nullptr;
  if (il) {
    const size_t hb = (size_t)ws.rows_p * h * sizeof(__half);
    const size_t qb = il_q8_bytes(ws.rows_p, h);
    // the padding half of a lone last half group (hidden_dim % 16 == 8) must read as zero in BOTH plane buffers: the epilogue
    // rewrites it as zero every iteration, the entry conversion below only writes the valid halves
    // (resume: nothing to convert, and both padding halves were zeroed by the call that started the sequence)
    if (!resume && h % 16 != 0) IADMM_CUDA(cudaMemsetAsync(ws.tc.h_lo[1], 0, qb, st));
    if (resume) {
    } else if (flags & IADMM_F_ZERO_STATE) {
      IADMM_CUDA(cudaMemsetAsync(ws.tc.h_hi[0], 0, hb, st));
      IADMM_CUDA(cudaMemsetAsync(ws.tc.h_lo[0], 0, qb, st));
      IADMM_CUDA(cudaMemsetAsync(ws.c_il, 0, (size_t)ws.rows_p * h * sizeof(float), st));
    } else {
      if (h % 16 != 0) IADMM_CUDA(cudaMemsetAsync(ws.tc.h_lo[0], 0, qb, st));
      if ((rc = launch_split_state_il(H, ws.tc.h_hi[0], ws.tc.h_lo[0], rows, h, st))) return rc;
      if ((rc = launch_c_to_il(C, ws.c_il, rows, h, st))) return rc;
    }
  } else if (tc) {
    if (flags & IADMM_F_ZERO_STATE) rc = launch_zero_state(ws.tc.h_hi[0], ws.tc.h_lo[0], rows, h, gp.nprod, st);
    else                            rc = launch_split_state(H, ws.tc.h_hi[0], ws.tc.h_lo[0], rows, h, gp.nprod, st);
    if (rc) return rc;
    // the other ping-pong buffer: padding bytes of the packed e4m3 rows must be finite (never multiplied, but loaded)
    if (gp.nprod == 2 && K > 1) IADMM_CUDA(cudaMemsetAsync(ws.tc.h_lo[1], 0, tc_lo_bytes(rows, h), st));
  }
  // programmatic dependent launches inside the KKT phase (common.cuh): measured, bit-identical and NOT faster (KKT phase 0.652 vs
  // 0.652 ms, 1.528 vs 1.522 ms at n = 5000, profiles/r02_kkt_pdl_ab.jsonl: the kernel boundaries are not where the phase loses
  // time), so plain launches stay the default and this is a development switch.  Pass 1 of iteration k > 0 follows this call's
  // own tail kernel, so nothing it reads before its wait (Q, A0) was written by its predecessor; iteration 0 is always launched
  // normally (the kernel before it may be the Ruiz scaling that wrote Q and A0).
  const char* pdl_sw = dev_env("IADMM_PDL");               // development switch: 1 = programmatic dependent launches
  const bool pdl = pdl_sw && pdl_sw[0] == '1';
  for (int k = 0; k < K; ++k) {
    const Sched* sk = sched + (t0 + k);
    prof_begin(kProfKkt, st);
    if ((rc = launch_kkt_pass1(ws.d, Q, A0, xv, x, y, ws.s, st, sp, pdl && k > 0))) return rc;
    if ((rc = launch_kkt_combine1(ws.d, p, xv, x, y, z, sk, sigma, ws.s, pri_trace, dual_trace, pri_trace_u,
                                  dual_trace_u, sd, se, sc, (k > 0 && want_trace) ? k - 1 : -1, 0, st, metric_trace, zu,
                                  k > 0 ? sk - 1 : nullptr, pdl))) return rc;
    if ((rc = launch_kkt_pass2(ws.d, Q, A0, ws.s, st, sp, pdl))) return rc;
    if ((rc = launch_kkt_combine2(ws.d, sk, sigma, ws.s, st, pdl))) return rc;
    prof_end(kProfKkt, st);
    prof_begin(kProfGates, st);
    if (tc) {
      ilp.C_rm_out = (k == K - 1) ? C : nullptr;
      rc = launch_gates_tc(packed_weights, L, xv, ws.s.g, ws.tc.h_hi[cur], ws.tc.h_lo[cur], ws.tc.h_hi[cur ^ 1],
                           ws.tc.h_lo[cur ^ 1], (k == K - 1) ? H : nullptr, C, ws.head_part, rows, h, gp, st, nullptr,
                           il ? &ilp : nullptr);
    } else {
      rc = launch_gates_simt(packed_weights, L, xv, ws.s.g, hbuf[cur], hbuf[cur ^ 1], C, ws.head_part, rows, h, st);
    }
    if (rc) return rc;
    prof_end(kProfGates, st);
    prof_begin(kProfTail, st);
    cur ^= 1;
    if ((rc = launch_tail(ws.d, ws.head_part, gp.head_slots, b_h, sk, zl, zu, x, y, z, xv, st, metric_trace ? &ws.s : nullptr))) return rc;
    prof_end(kProfTail, st);
  }
  if (!tc && cur == 1)
    IADMM_CUDA(cudaMemcpyAsync(H, ws.h_alt, (size_t)rows * h * sizeof(float), cudaMemcpyDeviceToDevice, st));
  if (want_trace && !(flags & IADMM_F_SKIP_FINAL_RESID)) {
    if ((rc = launch_kkt_pass1(ws.d, Q, A0, xv, x, y, ws.s, st, sp))) return rc;
    if ((rc = launch_kkt_combine1(ws.d, p, xv, x, y, z, nullptr, sigma, ws.s, pri_trace, dual_trace, pri_trace_u,
                                  dual_trace_u, sd, se, sc, K - 1, 1, st, metric_trace, zu, sched + (t0 + K - 1)))) return rc;
  }
  return IADMM_OK;
}

int iadmm_solve_state_resumable(int n, int m, int h, int mode, int flags, int* yes) {
  if (n <= 0 || m < 0 || h <= 0 || !yes) IADMM_FAIL(IADMM_ESHAPE, "solve_state_resumable: n=%d m=%d h=%d", n, m, h);
  // IADMM_F_KEEP_PLANES asks for the row-interleaved planes wherever a path has them; an unsupported mode or shape has none
  GatePlan gp;
  *yes = (plan_gates(mode, h, n, m, 1, flags | IADMM_F_KEEP_PLANES, false, &gp) == IADMM_OK && gp.interleaved) ? 1 : 0;
  return IADMM_OK;
}

int iadmm_solve(const void* packed_weights, const float* Q, const float* p, const float* A0, const float* zl,
                const float* zu, const float* sd, const float* se, const float* sc, float* x, float* y, float* z,
                float* xv, float* H, float* C, float* pri_trace, float* dual_trace, float* pri_trace_u,
                float* dual_trace_u, float* metric_trace, int B, int n, int num_ineq, int num_eq, int h, int length, int t0, int K,
                float sigma, int mode, int flags, void* workspace, size_t workspace_bytes, void* stream) {
  return solve_impl(packed_weights, Q, p, A0, zl, zu, sd, se, sc, x, y, z, xv, H, C, pri_trace, dual_trace, pri_trace_u, dual_trace_u,
                    metric_trace, B, n, num_ineq, num_eq, h, length, t0, K, sigma, mode, flags, workspace, workspace_bytes, stream,
                    nullptr);
}

int iadmm_solve_sparse(const void* packed_weights, const float* Q, const void* Q_sparse, size_t q_cap, const void* Q_blocks,
                       const float* p, const float* A0, const void* A0_sparse, size_t a_cap, const void* A0_blocks,
                       const float* zl, const float* zu,
                       const float* sd, const float* se, const float* sc, float* x, float* y, float* z,
                       float* xv, float* H, float* C, float* pri_trace, float* dual_trace, float* pri_trace_u,
                       float* dual_trace_u, float* metric_trace, int B, int n, int num_ineq, int num_eq, int h, int length, int t0,
                       int K, float sigma, int mode, int flags, void* workspace, size_t workspace_bytes, void* stream) {
  if (B <= 0 || n <= 0 || num_ineq < 0 || num_eq < 0) IADMM_FAIL(IADMM_ESHAPE, "solve_sparse: B=%d n=%d ineq=%d eq=%d", B, n, num_ineq, num_eq);
  if (!Q_sparse && !A0_sparse && !Q_blocks && !A0_blocks)
    IADMM_FAIL(IADMM_EALIGN, "solve_sparse: neither matrix is given in sparse form (use iadmm_solve)");
  if ((Q_sparse && Q_blocks) || (A0_sparse && A0_blocks)) IADMM_FAIL(IADMM_EMODE, "solve_sparse: one sparse form per matrix");
  if ((Q_sparse && !aligned16(Q_sparse)) || (A0_sparse && !aligned16(A0_sparse)) || (Q_blocks && !aligned16(Q_blocks)) ||
      (A0_blocks && !aligned16(A0_blocks)))
    IADMM_FAIL(IADMM_EALIGN, "solve_sparse: sparse buffers must be 16-byte aligned");
  if ((Q_blocks && !Q) || (A0_blocks && !A0)) IADMM_FAIL(IADMM_EALIGN, "solve_sparse: the block-skip form reads the dense matrix");
  KktSparse sp;
  memset(&sp, 0, sizeof(sp));
  const int m_ = num_ineq + num_eq;
  if (Q_sparse) sparse_view(Q_sparse, B, n, n, q_cap, &sp.q);
  if (A0_sparse && m_ > 0) sparse_view(A0_sparse, B, m_, n, a_cap, &sp.a);
  if (Q_blocks) { sp.q.blk = static_cast<const unsigned long long*>(Q_blocks); sp.q.blk_stride = (size_t)(n + 7) / 8; }
  if (A0_blocks && m_ > 0) { sp.a.blk = static_cast<const unsigned long long*>(A0_blocks); sp.a.blk_stride = (size_t)(m_ + 7) / 8; }
  return solve_impl(packed_weights, Q, p, A0, zl, zu, sd, se, sc, x, y, z, xv, H, C, pri_trace, dual_trace, pri_trace_u, dual_trace_u,
                    metric_trace, B, n, num_ineq, num_eq, h, length, t0, K, sigma, mode, flags | IADMM_F_STREAMING, workspace,
                    workspace_bytes, stream, &sp);
}

int iadmm_profile_begin(int max_iterations) {
  if (max_iterations <= 0 || max_iterations > (1 << 20)) IADMM_FAIL(IADMM_ESHAPE, "profile_begin: max_iterations=%d", max_iterations);
  if (g_prof.span) IADMM_FAIL(IADMM_ESHAPE, "profile_begin: a profile is already open");
  const size_t cap = (size_t)max_iterations * 8;       // at most 8 spans per iteration (3 in the solve, 7 in a training iteration)
  g_prof.span = new ProfSpan[cap];
  for (size_t i = 0; i < cap; ++i) {
    IADMM_CUDA(cudaEventCreate(&g_prof.span[i].e0));
    IADMM_CUDA(cudaEventCreate(&g_prof.span[i].e1));
  }
  for (int k = 0; k < kProfKinds; ++k) g_prof.open[k] = -1;
  g_prof.cap = (int)cap; g_prof.used = 0; g_prof.on = true;
  return IADMM_OK;
}

int iadmm_profile_end_kinds(double* ms_by_kind, int* spans_by_kind, int kinds) {
  if (!g_prof.span) IADMM_FAIL(IADMM_ESHAPE, "profile_end: no open profile");
  if (kinds < 0 || kinds > kProfKinds) IADMM_FAIL(IADMM_ESHAPE, "profile_end: kinds=%d (the library records %d)", kinds, kProfKinds);
  g_prof.on = false;
  double ms[kProfKinds] = {0};
  int cnt[kProfKinds] = {0};
  int rc = IADMM_OK;
  // every recorded event must have completed: wait for the device once (measurement code, not the hot path)
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { set_error("profile_end: %s", cudaGetErrorString(e)); rc = IADMM_ECUDA; }
  for (int i = 0; i < g_prof.used && rc == IADMM_OK; ++i) {
    float t = 0.f;
    if (cudaEventElapsedTime(&t, g_prof.span[i].e0, g_prof.span[i].e1) == cudaSuccess) {   // fails for a span that was never closed
      ms[g_prof.span[i].kind] += t;
      ++cnt[g_prof.span[i].kind];
    }
  }
  (void)cudaGetLastError();
  for (int i = 0; i < g_prof.cap; ++i) { cudaEventDestroy(g_prof.span[i].e0); cudaEventDestroy(g_prof.span[i].e1); }
  delete[] g_prof.span;
  g_prof.span = nullptr;
  g_prof.cap = g_prof.used = 0;
  for (int k = 0; k < kinds; ++k) {
    if (ms_by_kind) ms_by_kind[k] = ms[k];
    if (spans_by_kind) spans_by_kind[k] = cnt[k];
  }
  return rc;
}

int iadmm_profile_end(double* kkt_ms, double* gates_ms, double* tail_ms, int* iterations) {
  double ms[kProfKinds];
  int cnt[kProfKinds];
  int rc = iadmm_profile_end_kinds(ms, cnt, kProfKinds);
  if (rc) return rc;
  if (kkt_ms) *kkt_ms = ms[kProfKkt];
  if (gates_ms) *gates_ms = ms[kProfGates];
  if (tail_ms) *tail_ms = ms[kProfTail];
  if (iterations) *iterations = cnt[kProfGates];
  return IADMM_OK;
}

int iadmm_residuals_workspace_bytes(int B, int n, int m, size_t* bytes) {
  if (B <= 0 || n <= 0 || m < 0 || !bytes) IADMM_FAIL(IADMM_ESHAPE, "residuals_workspace_bytes: B=%d n=%d m=%d", B, n, m);
  *bytes = kkt_scratch_floats(make_kkt_dims(B, n, m, 0)) * sizeof(float);
  return IADMM_OK;
}

int iadmm_residuals(const float* x, const float* y, const float* z, const float* Q, const float* p, const float* A0,
                    float* pri, float* dual, int B, int n, int m, void* workspace, size_t workspace_bytes,
                    void* stream) {
  if (B <= 0 || n <= 0 || m < 0) IADMM_FAIL(IADMM_ESHAPE, "residuals: B=%d n=%d m=%d", B, n, m);
  if (B > 65535) IADMM_FAIL(IADMM_ESHAPE, "residuals: batch %d > 65535 per call", B);
  if (!x || !Q || !p || !pri || !dual || !workspace) IADMM_FAIL(IADMM_EALIGN, "residuals: NULL pointer");
  if (m > 0 && (!y || !z || !A0)) IADMM_FAIL(IADMM_EALIGN, "residuals: NULL constraint pointer");
  int rc = check_device();
  if (rc) return rc;
  const KktDims d = make_kkt_dims(B, n, m, 0);
  if (kkt_scratch_floats(d) * sizeof(float) > workspace_bytes) IADMM_FAIL(IADMM_EWORK, "residuals: workspace too small");
  KktScratch s;
  kkt_scratch_carve(d, static_cast<float*>(workspace), &s);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if ((rc = launch_kkt_pass1_plain(d, Q, A0, x, y, s, st))) return rc;
  return launch_kkt_combine1(d, p, nullptr, x, y, z, nullptr, 0.f, s, pri, dual, nullptr, nullptr, nullptr, nullptr,
                             nullptr, 0, 1, st);
}

int iadmm_kkt_penalty_diagonal(const void* packed_weights, float* Kmat, int B, int n, int num_ineq, int num_eq, int h,
                               int length, int t, void* stream) {
  const int m = num_ineq + num_eq;
  if (B <= 0 || n <= 0 || m < 0 || t < 0 || t >= length) IADMM_FAIL(IADMM_ESHAPE, "kkt_penalty_diagonal: B=%d n=%d m=%d t=%d length=%d", B, n, m, t, length);
  if (!packed_weights || !Kmat) IADMM_FAIL(IADMM_EALIGN, "kkt_penalty_diagonal: NULL pointer");
  int rc = check_device();
  if (rc) return rc;
  const WeightLayout L = weight_layout(h, length);
  const Sched* sched = reinterpret_cast<const Sched*>(static_cast<const char*>(packed_weights) + L.off_sched) + t;
  return launch_kkt_penalty_diag(B, n, m, num_ineq, sched, Kmat, static_cast<cudaStream_t>(stream));
}

int iadmm_build_kkt(const void* packed_weights, const float* Q, const float* p, const float* A0, const float* x,
                    const float* y, const float* z, float* Kmat, float* rhs, float* rho_vec, int B, int n,
                    int num_ineq, int num_eq, int h, int length, int t, float sigma, void* stream) {
  const int m = num_ineq + num_eq;
  if (B <= 0 || n <= 0 || m < 0 || t < 0 || t >= length) IADMM_FAIL(IADMM_ESHAPE, "build_kkt: B=%d n=%d m=%d t=%d length=%d", B, n, m, t, length);
  if (B > 65535 || n + m > 65535) IADMM_FAIL(IADMM_ESHAPE, "build_kkt: B and n+m must be <= 65535");
  if (!packed_weights || !Q || !p || !x || !rhs) IADMM_FAIL(IADMM_EALIGN, "build_kkt: NULL pointer");
  int rc = check_device();
  if (rc) return rc;
  const WeightLayout L = weight_layout(h, length);
  const Sched* sched = reinterpret_cast<const Sched*>(static_cast<const char*>(packed_weights) + L.off_sched) + t;
  return launch_build_kkt(B, n, m, num_ineq, Q, p, A0, x, y, z, sched, sigma, Kmat, rhs, rho_vec,
                          static_cast<cudaStream_t>(stream));
}

}  // extern "C"

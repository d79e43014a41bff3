/*
 * iadmm.h -- C ABI of libiadmm_b200.so: the B200 (sm_100a) implementation of the I-ADMM-LSTM
 * unrolled solve path.
 *
 * The reference (NetSysOpt/I-ADMM-LSTM) has no FFI layer; its boundary for this path is three Python
 * call signatures.  Each entry point below names the reference interface it replaces (paths relative
 * to the reference checkout).  INTEGRATION.md shows the ctypes binding a maintainer adds on the
 * reference side.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to contiguous fp32 memory owned by the caller, 16-byte aligned
 *     (torch allocations are 256-byte aligned); the library never allocates or frees caller-visible
 *     memory; between calls it keeps only the last error string (thread local), per-device caches of
 *     immutable facts (SM count, per-kernel shared-memory opt-in) and a per-thread cache of TMA descriptors
 *     keyed by (address, shape) -- nothing that depends on buffer contents.  One process may drive several
 *     devices (cudaSetDevice before the call, as torch.cuda.device() does);
 *   - the release build reads NO environment variable (development switches exist only in
 *     libiadmm_b200_dev.so, built with IADMM_DEV_BUILD=1);
 *   - vectors are the reference's [B, dim, 1] columns, i.e. [B, dim] contiguous; matrices are
 *     row-major [B, rows, cols]; rows of A0 are the num_ineq inequality rows, then the num_eq
 *     equality rows (generate_data.py:74);
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued asynchronously on it and
 *     nothing synchronises the device;
 *   - return value 0 = success, negative = IADMM_E*; iadmm_last_error() describes the failure.
 *     There is no CPU fallback: on a device that is not compute capability 10.x every compute
 *     entry point fails with IADMM_EARCH.
 */
#ifndef IADMM_H_
#define IADMM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IADMM_ABI_VERSION 3

enum {
  IADMM_OK      = 0,
  IADMM_ESHAPE  = -1,   /* negative / inconsistent sizes, t0+K > schedule length */
  IADMM_EALIGN  = -2,   /* pointer not 16-byte aligned or NULL where required */
  IADMM_EARCH   = -3,   /* current device is not sm_100 */
  IADMM_ECUDA   = -4,   /* a CUDA runtime/driver call failed (message has the cudaError) */
  IADMM_EWORK   = -5,   /* workspace too small */
  IADMM_EMODE   = -6    /* unknown or unsupported mode for these sizes */
};

/* Gate-contraction arithmetic (models/lstm.py:74-77, the [B*N,h]x[h,4h] product H_t @ U_*). */
enum {
  IADMM_GATES_SIMT_FP32   = 0,  /* fp32 FMA on CUDA cores: bit-stable validation path                   */
  IADMM_GATES_TC_3XFP16   = 1,  /* tcgen05, fp16 hi/lo split of both operands, 3 MMAs, fp32 accumulate: */
                                /* ~22-bit operands (parity <= 1e-4 after K=100)                        */
  IADMM_GATES_TC_1XFP16   = 2,  /* tcgen05, single fp16 MMA (TF32-class operands): opt-in fast mode     */
  IADMM_GATES_TC_F16F8    = 3,  /* tcgen05, fp16 main product + two fp8 (e4m3) correction products for  */
                                /* the operand rounding residuals: ~16-bit operands at 2/3 of the cost  */
                                /* of the 3-way split: THE DEFAULT.  hidden_dim % 8 == 0; with           */
                                /* hidden_dim % 16 == 8 (configs/QP.yaml's 200) the solve pads the last */
                                /* 16-unit operand group, training uses the 3-way split                  */
  IADMM_GATES_TC_F16F8U   = 4   /* opt-in: as F16F8, but wherever the solve keeps its state             */
                                /* row-interleaved only the rounding of the WEIGHTS U is corrected (1.5 */
                                /* instead of 2 MMA units): the HBM-streaming solve with K >= 2, with   */
                                /* hidden_dim % 16 == 8, or with IADMM_F_KEEP_PLANES / IADMM_F_RESUME   */
                                /* (LSTM.forward's steps on that path).  The on-chip-resident solve,    */
                                /* the other K = 1 calls and training run F16F8 exactly.  The fp16      */
                                /* rounding of H then acts as fresh 2^-12 noise every iteration: K=100  */
                                /* parity measured at 1e-5..5e-5, inside the 1e-4 bar with a 2x (not    */
                                /* 20x) margin -- see DESIGN.md                                         */
};

/* Flags of iadmm_solve. */
enum {
  IADMM_F_ZERO_STATE = 1,       /* H (and the other state) is known to be all-zero on entry (main.py:837-843) */
  IADMM_F_SKIP_FINAL_RESID = 2, /* do not run the trailing residual pass (traces row K-1 left untouched)      */
  IADMM_F_STREAMING = 4,        /* force the streaming (HBM) variant even where the on-chip-resident one applies  */
  /* The reference drives the path ONE iteration per call (main.py:874-887: model(t, ...) with the returned H, C fed
   * back).  The next three flags let such a loop run without converting H and C between the caller's fp32 tensors
   * and the kernels' row-interleaved operand planes on every call (iadmm_solve_state_resumable says when they apply): */
  IADMM_F_KEEP_PLANES = 8,      /* keep the state in the row-interleaved planes of the workspace even for K = 1, so   */
                                /* that the NEXT call on the same workspace can resume from them                      */
  IADMM_F_RESUME = 16,          /* H and C on entry are NOT read: the state is taken from the planes the previous     */
                                /* call (same workspace, B, n, m, h, mode; workspace untouched since) left behind.    */
                                /* H and C are still fully written on exit.  Implies IADMM_F_KEEP_PLANES              */
  IADMM_F_RESUME_ODD = 32       /* with IADMM_F_RESUME: the planes are in ping-pong buffer 1.  A call that runs K     */
                                /* iterations from buffer c leaves them in buffer (c + K) & 1 (c = 0 without RESUME)  */
};

int         iadmm_abi_version(void);
const char* iadmm_last_error(void);
/* 0 if the CURRENT cuda device can run the kernels (compute capability 10.x), else IADMM_EARCH/ECUDA. */
int         iadmm_device_check(void);

/* ---- weights ------------------------------------------------------------------------------------
 * Replaces: the 16 nn.Parameters of models/lstm.py:21-41 as consumed by LSTM.forward (:60-63, :74-80).
 * Packs them once per weight update into the layouts the kernels read:
 *   - U_{i,f,o,u} interleaved per hidden unit (column 4*j+g), as fp32 [h][4h] and as fp16 hi/lo
 *     K-major [4*h_pad][h_pad] tiles for the tensor-core path,
 *   - W rows, biases, W_h, b_h,
 *   - the schedule rho_t = sigmoid(rho[t]), 1e3*rho_t, their reciprocals, alpha_t = 2*sigmoid(alpha[t]).
 * `packed` must hold iadmm_weights_bytes(h, length) bytes.
 */
int iadmm_weights_bytes(int h, int length, size_t* bytes);
int iadmm_pack_weights(const float* W_i, const float* U_i, const float* b_i,
                       const float* W_f, const float* U_f, const float* b_f,
                       const float* W_o, const float* U_o, const float* b_o,
                       const float* W_u, const float* U_u, const float* b_u,
                       const float* W_h, const float* b_h,
                       const float* rho, const float* alpha,
                       int h, int length, void* packed, void* stream);

/* ---- Ruiz equilibration -------------------------------------------------------------------------
 * Replaces: Scaling.scale_data, methods/scaling.py:50-119 (incl. _norm_KKT_cols :17-29 and
 * _limit_scaling :31-46).  O(n^2) streaming passes on the diagonals instead of dense diag bmm's;
 * element-wise products are rounded in the reference's order, so outputs match it bit-for-bit up to
 * the summation order of one mean per iteration.
 * In : Q [B,n,n], p [B,n], A0 [B,m,n], zl, zu [B,m]  (zl may hold -inf, zu +inf).
 * Out: Qs, ps, A0s, zls, zus (same shapes, may NOT alias the inputs), d [B,n], e [B,m], c [B]
 *      with D = diag(d), E = diag(e) (scaling.py:107-117).
 */
int iadmm_ruiz_workspace_bytes(int B, int n, int m, size_t* bytes);
int iadmm_ruiz(const float* Q, const float* p, const float* A0, const float* zl, const float* zu,
               float* Qs, float* ps, float* A0s, float* zls, float* zus,
               float* d, float* e, float* c,
               int B, int n, int m, int iterations,
               void* workspace, size_t workspace_bytes, void* stream);

/* ---- the unrolled solve -------------------------------------------------------------------------
 * Replaces: K consecutive calls of LSTM.forward (models/lstm.py:47-96) as driven by main.py:874-887
 * (test), :338-347 (train forward) and :503-509 (validation), plus the residual evaluation
 * primal_dual_loss (utils.py:68-71) main.py performs after every call (:346, :955).
 *
 * State x [B,n], y,z [B,m], xv [B,n+m], H,C [B,n+m,h] is updated IN PLACE (iterations t0..t0+K-1 of
 * the schedule).  Traces are [K,B] row-major, optional (NULL to skip):
 *   pri_trace/dual_trace     residuals on the data passed in                       (main.py:346)
 *   pri_trace_u/dual_trace_u residuals of the un-scaled iterates on the original data, computed from
 *                            the diagonals d,e,c of iadmm_ruiz (main.py:922-955); need d,e,c != NULL.
 *   metric_trace             [K,6,B]: objective 0.5 x^T Q x + p^T x (utils.py:53), max and mean of relu(G x - c)
 *                            over the inequality rows (utils.py:56) and of |b - A x| over the equality rows
 *                            (utils.py:59), i.e. the per-instance quantities main.py:949-968 prints; evaluated on
 *                            the original data when d,e,c are given (with the un-scaled iterate), else on the
 *                            data passed in.  Row 5: the linear-system residual ||A_tild xv - b_tild|| of
 *                            main.py:952 (K and rhs of the iteration that produced xv, on the data passed in).
 * mode: IADMM_GATES_*; flags: IADMM_F_*.
 */
int iadmm_solve_workspace_bytes(int B, int n, int m, int h, int mode, size_t* bytes);
/* *yes = 1 when iadmm_solve honours IADMM_F_KEEP_PLANES / IADMM_F_RESUME for this shape and mode (the fp16+fp8 modes on the
 * HBM-streaming path), else 0: IADMM_F_KEEP_PLANES is then ignored and H, C are read on entry as usual; IADMM_F_RESUME is
 * ignored by the on-chip-resident path and rejected with IADMM_EMODE elsewhere. */
int iadmm_solve_state_resumable(int n, int m, int h, int mode, int flags, int* yes);
int iadmm_solve(const void* packed_weights,
                const float* Q, const float* p, const float* A0, const float* zl, const float* zu,
                const float* d, const float* e, const float* c,
                float* x, float* y, float* z, float* xv, float* H, float* C,
                float* pri_trace, float* dual_trace, float* pri_trace_u, float* dual_trace_u,
                float* metric_trace,
                int B, int n, int num_ineq, int num_eq, int h, int length, int t0, int K,
                float sigma, int mode, int flags,
                void* workspace, size_t workspace_bytes, void* stream);

/* ---- sparse problem families ----------------------------------------------------------------------
 * Replaces: the `.toarray()` densification of main.py:243-296 for the families generate_data.py:96-228 stores as scipy
 * csc matrices (Random_QP: A0 60 % dense; Equality_QP: 50 %; SVM: identity blocks) and the QPLIB / Maros-Meszaros
 * instances.  iadmm_sparse_pack re-lays a dense [B, rows, n] batch (after Ruiz scaling, which keeps the pattern) as
 * "bitmap slabs": per row and 128-column slab a 128-bit occupancy mask and the offset of its first value, plus the
 * instance's non-zero values in row-major order -- 4*nnz + 20*rows*ceil(n/128) bytes per instance instead of 4*rows*n.
 * `cap` = value capacity per instance (>= the largest instance's non-zero count; rows*n always suffices); `nnz` (device,
 * [B], may be NULL) receives the counts -- values beyond `cap` are NOT stored, so check max(nnz) <= cap.
 * iadmm_solve_sparse = iadmm_solve with Q and/or A0 given in that form (pass NULL for the form not used; the dense
 * pointer of a matrix given in sparse form may be NULL).  Same kernels, same lane-to-column assignment and accumulation
 * order as the dense passes: results are bit-identical to the densified problem, the KKT passes read only the stored bytes.
 * Always runs the HBM-streaming variant.
 *
 * Second form, for STRUCTURED sparsity (diagonal Q of the QP family, the identity blocks of SVM, banded QPLIB matrices):
 * the dense matrix stays as it is and iadmm_block_mask computes one bit per 8-row x 128-column block ("does it hold a
 * non-zero"): blocks [B][ceil(rows/8)] 64-bit words, bit s of word g <-> rows 8g..8g+7, columns 128s..128s+127 (n <= 8192);
 * `nonempty` (device, [B], may be NULL) receives the number of non-empty blocks per instance.  A warp's unit of work in the
 * KKT passes IS such a block, so a clear bit skips its 4 KB of loads with a warp-uniform branch at no decode cost: HBM bytes
 * = the non-empty blocks, results bit-identical.  Pass the words as Q_blocks / A0_blocks (with the dense Q / A0).  The
 * bitmap-slab form wins below ~0.3 % density on unstructured patterns, block skipping whenever whole blocks are empty;
 * unstructured 1-60 % dense matrices are fastest in plain dense form (the mask expansion is instruction bound). */
int iadmm_sparse_bytes(int B, int rows, int n, size_t cap, size_t* bytes);
int iadmm_sparse_pack(const float* M, int B, int rows, int n, size_t cap, void* packed, size_t packed_bytes, int* nnz,
                      void* stream);
int iadmm_block_mask_bytes(int B, int rows, int n, size_t* bytes);
int iadmm_block_mask(const float* M, int B, int rows, int n, void* blocks, size_t blocks_bytes, unsigned int* nonempty,
                     void* stream);
int iadmm_solve_sparse(const void* packed_weights,
                       const float* Q, const void* Q_sparse, size_t q_cap, const void* Q_blocks, const float* p,
                       const float* A0, const void* A0_sparse, size_t a_cap, const void* A0_blocks,
                       const float* zl, const float* zu,
                       const float* d, const float* e, const float* c,
                       float* x, float* y, float* z, float* xv, float* H, float* C,
                       float* pri_trace, float* dual_trace, float* pri_trace_u, float* dual_trace_u,
                       float* metric_trace,
                       int B, int n, int num_ineq, int num_eq, int h, int length, int t0, int K,
                       float sigma, int mode, int flags,
                       void* workspace, size_t workspace_bytes, void* stream);

/* ---- adjacent pieces of the reference interface ------------------------------------------------- */

/* Replaces: primal_dual_loss, utils.py:68-71 (forward).  pri, dual: [B]. */
int iadmm_residuals_workspace_bytes(int B, int n, int m, size_t* bytes);
int iadmm_residuals(const float* x, const float* y, const float* z,
                    const float* Q, const float* p, const float* A0,
                    float* pri, float* dual, int B, int n, int m,
                    void* workspace, size_t workspace_bytes, void* stream);

/* Replaces: the A_tild / b_tild / rho_vec members of LSTM.forward's return tuple
 * (models/lstm.py:61-62, :67-69, :96), which main.py:952 and the Stage-II solver (models/lu.py) read.
 * The solve itself never forms them.  Kmat [B,n+m,n+m] (NULL: only rhs and rho_vec, O(n+m) work),
 * rhs [B,n+m], rho_vec [B,m]; x,y,z are the iterates BEFORE iteration t. */
int iadmm_build_kkt(const void* packed_weights, const float* Q, const float* p, const float* A0,
                    const float* x, const float* y, const float* z,
                    float* Kmat, float* rhs, float* rho_vec,
                    int B, int n, int num_ineq, int num_eq, int h, int length, int t, float sigma,
                    void* stream);
/* Rewrites the -(1/rho_t) diagonal of the last m rows of a Kmat that iadmm_build_kkt produced for the same Q, A0 and sigma at
 * another iteration: the only entries of A_tild that depend on t (models/lstm.py:60-62, :68).  Lets a caller keep ONE dense
 * A_tild per problem batch over the per-iteration loop of main.py:874-887 instead of writing 4(n+m)^2 bytes per call. */
int iadmm_kkt_penalty_diagonal(const void* packed_weights, float* Kmat, int B, int n, int num_ineq, int num_eq,
                               int h, int length, int t, void* stream);

/* ---- Stage II (feasibility restoration): batched dense LU --------------------------------------------
 * Replaces: `torch.lu(A_tild, pivot=True)` (models/lu.py:30) -- LAPACK getrf semantics, partial pivoting,
 * first maximum.  Kmat [B,N,N] row-major is overwritten by L (unit, below the diagonal) and U; piv [B,N] is
 * the 0-based interchange sequence, perm [B,N] the resulting row permutation (row i of P*K = row perm[i] of
 * K), info [B] (may be NULL) is 0 or 1 + the index of the first exactly-zero pivot.  N <= 4096 (its 16-column
 * panel is held in the registers of one CTA); larger systems go to iadmm_lu_factor_blocked. */
int iadmm_lu_factor(float* Kmat, int* piv, int* perm, int* info, int B, int N, void* stream);

/* The same factorisation for 1 <= N <= 32768 (B <= 65535), with the same outputs and semantics, so iadmm_lu_solve
 * consumes them unchanged.  Blocked right-looking LU with 128-column outer blocks: each 16-column sub-panel runs on a
 * thread-block cluster of up to 8 CTAs (4096 rows each) that agree on every pivot through distributed shared memory;
 * the trailing update A22 -= L21 U12 runs on the tensor cores as three tf32 products (hi*hi + hi*lo + lo*hi of a tf32
 * hi/lo split of both operands, fp32 accumulation), ~fp32 accuracy without scaling.  Results are deterministic, but
 * not bit-identical to iadmm_lu_factor's (the update order differs).  `workspace` holds the split operands; its size
 * comes from iadmm_lu_factor_blocked_workspace_bytes and its contents on entry do not matter.
 * Errors: IADMM_EMODE for N > 32768, IADMM_EWORK for a short workspace, IADMM_EALIGN for NULL pointers (info may be
 * NULL), IADMM_EARCH off sm_100. */
int iadmm_lu_factor_blocked_workspace_bytes(int B, int N, size_t* bytes);
int iadmm_lu_factor_blocked(float* Kmat, int* piv, int* perm, int* info, int B, int N,
                            void* workspace, size_t workspace_bytes, void* stream);

/* Replaces: `torch.lu_solve(b_tild, lu, piv)` (models/lu.py:35), once per Stage-II iteration.
 * rhs [B,N] is overwritten by the solution. */
int iadmm_lu_solve(const float* LU, const int* perm, float* rhs, int B, int N, void* stream);

/* ---- training: truncated BPTT through the unroll -------------------------------------------------------
 * Replaces: the autograd tape PyTorch records through LSTM.forward (models/lstm.py:47-96) and
 * primal_dual_loss (utils.py:68-71) in the training loop main.py:336-358.  One differentiable iteration =
 * iadmm_step_fwd (out of place, saves g = K^T(K xv - rhs), w = K xv - rhs and the gate activations) +
 * iadmm_step_bwd (hand-written adjoint; reuses the two streaming KKT passes, two fp32 GEMMs for the gate
 * products).  The forward gate contraction runs in `mode` (IADMM_GATES_*, tensor cores by default like the solve;
 * F16F8 and F16F8U both keep the two correction products, as the 3-way split at hidden_dim % 16 == 8; a tensor-core mode
 * runs fp32 at hidden_dim % 8 != 0; an unknown mode is IADMM_EMODE); the backward's two gate-product GEMMs run on the
 * tensor cores at hidden_dim % 16 == 0 and in fp32 on CUDA cores otherwise.  Adam (main.py:191) stays in PyTorch;
 * data-parallel training all-reduces the flat gradient buffer over NCCL (iadmm_b200/dist.py).
 *
 * Every hidden_dim h >= 1 trains.  The kernels run the width hp = h rounded up to 4: for h % 4 != 0 each call re-lays the
 * weights and the state into the model of width hp whose extra units have zero parameters and a zero state, and the results
 * back.  Those units stay exactly zero (their gates are 0.5 and tanh(0)) and feed nothing into the real ones, so the outputs,
 * adjoints and gradients are bit for bit those of the zero-padded width-hp model, and every rule above applies at hp: e.g.
 * h = 50 runs the fp32 gates and backward of 52, h = 30 the tensor-core forward and backward of 32, h = 199 in tc_f16f8 the
 * 3-way split of 200.  The caller-facing shapes stay at h (H, C and their adjoints [B*(n+m), h], grad_flat in the layout of
 * iadmm_param_count(h, length), packed_weights the iadmm_pack_weights(h, length) image); the workspace-size queries include
 * the padded copies.
 *
 * grad_flat: [iadmm_param_count] floats in state_dict order (W_i,U_i,b_i, W_f,.., W_u,U_u,b_u, W_h, b_h, rho,
 * alpha); iadmm_step_bwd ADDS this iteration's parameter adjoints to it.  Incoming adjoints g*_o may be
 * NULL (= zero); outgoing adjoints gx..gC are overwritten.  gates_save: [B*(n+m), 4*hp] (NULL in iadmm_step_fwd: not kept),
 * i.e. [B*(n+m), 4h] whenever h % 4 == 0.
 */
int iadmm_param_count(int h, int length, size_t* count);
int iadmm_train_workspace_bytes(int B, int n, int m, int h, size_t* bytes);
int iadmm_step_fwd(const void* packed_weights,
                   const float* Q, const float* p, const float* A0, const float* zl, const float* zu,
                   const float* x, const float* y, const float* z, const float* xv, const float* H, const float* C,
                   float* x_o, float* y_o, float* z_o, float* xv_o, float* H_o, float* C_o,
                   float* g_save, float* w_save, float* gates_save,
                   int B, int n, int num_ineq, int num_eq, int h, int length, int t, float sigma, int mode,
                   void* workspace, size_t workspace_bytes, void* stream);
int iadmm_step_bwd(const void* packed_weights,
                   const float* Q, const float* p, const float* A0, const float* zl, const float* zu,
                   const float* x, const float* y, const float* z, const float* xv, const float* H, const float* C,
                   const float* xv_o, const float* H_o,
                   const float* g_save, const float* w_save, const float* gates_save,
                   const float* gx_o, const float* gy_o, const float* gz_o, const float* gxv_o,
                   const float* gH_o, const float* gC_o,
                   float* gx, float* gy, float* gz, float* gxv, float* gH, float* gC,
                   float* grad_flat,
                   int B, int n, int num_ineq, int num_eq, int h, int length, int t, float sigma,
                   void* workspace, size_t workspace_bytes, void* stream);
/* primal_dual_loss keeping r_p = A0 x - z [B,m] and r_d = Q x + p + A0^T y [B,n], and its adjoint
 * (gpri/gdual [B], NULL = zero). */
int iadmm_residuals_train_workspace_bytes(int B, int n, int m, size_t* bytes);
int iadmm_residuals_fwd(const float* x, const float* y, const float* z,
                        const float* Q, const float* p, const float* A0,
                        float* pri, float* dual, float* rp_save, float* rd_save,
                        int B, int n, int m, void* workspace, size_t workspace_bytes, void* stream);
int iadmm_residuals_bwd(const float* Q, const float* A0, const float* pri, const float* dual,
                        const float* rp_save, const float* rd_save, const float* gpri, const float* gdual,
                        float* gx, float* gy, float* gz,
                        int B, int n, int m, void* workspace, size_t workspace_bytes, void* stream);

/* One whole truncated-BPTT window (main.py:336-358) in a single call: for t = t0 .. t0+TL-1 the iteration
 * (iadmm_step_fwd) and primal_dual_loss on its output, loss = loss_scale * sum_t mean_b(pri_t + dual_t)
 * (loss_scale = 1/outer_T in main.py:347), then the backward sweep through the window.  x..C are updated in place to
 * the state after the window (the reference detaches it there, main.py:353-358); grad_flat [iadmm_param_count] is
 * OVERWRITTEN with d loss / d parameters (state_dict order, see above); loss_out [1].  Same kernels and results as
 * the per-iteration entry points, without the host round trips between them. */
enum { IADMM_TRAIN_RECOMPUTE_GATES = 1 };   /* flags of iadmm_train_window: do not keep the gate activations [TL, B*(n+m), 4hp] over
                                               the window; the backward re-runs the forward gate kernel per iteration on the saved
                                               H, C, xv, g (bit-identical activations, same gradients): 2.56 -> 0 GB per instance
                                               and window at n+m = 2000, hidden_dim 800, TL = 100, for one more gate product */
int iadmm_window_workspace_bytes(int B, int n, int m, int h, int TL, int flags, size_t* bytes);
int iadmm_train_window(const void* packed_weights,
                       const float* Q, const float* p, const float* A0, const float* zl, const float* zu,
                       float* x, float* y, float* z, float* xv, float* H, float* C,
                       float* grad_flat, float* loss_out,
                       int B, int n, int num_ineq, int num_eq, int h, int length, int t0, int TL, float sigma,
                       float loss_scale, int mode, int flags, void* workspace, size_t workspace_bytes, void* stream);

/* ---- data-parallel training: the one collective of the path ------------------------------------------
 * Replaces: nothing in the reference (single process); SURVEY.md section 8(b/e): one sum all-reduce of the flat gradient
 * buffer of iadmm_train_window / iadmm_step_bwd over NCCL (NVLink / NVSwitch) per truncated-BPTT window, in place, followed
 * by a multiplication with `scale` (1/world for equal shards; 1 when the caller weights the ranks itself).  `nccl_comm` is an
 * ncclComm_t passed as void*; NCCL is looked up in the host process at the first call (no link-time dependency). */
int iadmm_allreduce_grads(float* flat_grads, size_t count, float scale, void* nccl_comm, void* stream);
/* Communicator set-up without the host framework: rank 0 fills a 128-byte unique id (ncclGetUniqueId), the caller carries it to
 * the other ranks (any side channel), every rank joins with the CURRENT cuda device (ncclCommInitRank). */
int iadmm_nccl_unique_id(void* uid128);
int iadmm_nccl_comm_init(void** comm, int world, const void* uid128, int rank);
int iadmm_nccl_comm_destroy(void* comm);

/* ---- measurement hooks (bench.py) ------------------------------------------------------------------
 * The reference times its solve with time.time() around model() (main.py:881-890, no device sync).
 * Between iadmm_profile_begin and iadmm_profile_end every iadmm_solve call records CUDA events on its
 * own stream around the three phases of each iteration (KKT passes+combines | gate kernel | tail), up
 * to max_iterations iterations in total.  iadmm_profile_end synchronises on the last event and returns
 * the summed device time of each phase in milliseconds and the number of iterations recorded.
 * Process-wide, not thread safe; recording costs four event records per iteration. */
int iadmm_profile_begin(int max_iterations);
int iadmm_profile_end(double* kkt_ms, double* gates_ms, double* tail_ms, int* iterations);
/* Same, every span kind the library records: [0] KKT phase, [1] gate kernel, [2] tail of iadmm_solve; of the training
 * entry points [3] forward gate kernel, [4] the two gate-product adjoint GEMMs of the backward (with their operand
 * splits), [5] KKT passes (forward, residuals, adjoint), [6] cell adjoint and small parameter adjoints.
 * ms_by_kind / spans_by_kind: arrays of `kinds` (<= 7) entries, either may be NULL.  Synchronises the device. */
int iadmm_profile_end_kinds(double* ms_by_kind, int* spans_by_kind, int kinds);

#ifdef __cplusplus
}
#endif
#endif /* IADMM_H_ */

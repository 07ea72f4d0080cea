/*
 * sow_b200 -- C ABI of the B200-native SoW ("Sum-of-Weights", python package `tn_gradient`) training hot path.
 *
 * The reference (antoine311200/sow) is pure PyTorch and has no FFI of its own; its boundary for this path is the
 * Python surface of `tn_gradient` (SURVEY.md 8b).  This header is the boundary *underneath* that surface: every
 * entry point names the reference call site (file:line under the reference root) whose device math it replaces.
 *
 * Conventions
 *  - All pointers are BORROWED raw CUDA device pointers (except where marked host).  Nothing here allocates,
 *    frees, synchronises the device, or keeps a pointer after returning.
 *  - Every function returns 0 on success and a negative SOWB_E* code on failure; sow_last_error() returns a
 *    thread-local human-readable message for the last failure on the calling thread.
 *  - Work is enqueued on the caller's `stream` (a cudaStream_t passed as void*); calls are re-entrant and may be
 *    issued concurrently from several host threads (autograd runs backward on its own thread).
 *  - Scratch memory is provided by the caller: ask sow_workspace_bytes() first.
 *  - Matrices are dense row-major.  W is (in,out) -- the reference layout (tn_gradient/layer/sow.py:28,74-79),
 *    i.e. the transpose of nn.Linear.  dtype codes: SOWB_BF16 / SOWB_F32 / SOWB_F16.
 *  - 16-bit modes (SOWB_BF16, SOWB_F16): every 2-byte tensor of a call has the mode's type; products accumulate in fp32
 *    and every output element is rounded once to the 16-bit type (round to nearest even).  In SOWB_F16, values past
 *    65504 become +-inf and inf / NaN propagate (IEEE fp16, as torch's fp16 matmul; no saturation).
 *  - The tensor-train entry points (tt_*) take SOWB_BF16 / SOWB_F32 only and reject SOWB_F16 with SOWB_EINVAL.
 *  - Alignment: device pointers 16-byte aligned; `in` and `out` multiples of 8 (TMA row pitch rule).
 */
#ifndef SOW_B200_H_
#define SOW_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SOWB_OK 0
#define SOWB_EINVAL (-1)    /* bad argument (null pointer, unsupported shape/dtype, misalignment) */
#define SOWB_EWORKSPACE (-2) /* workspace too small */
#define SOWB_ECUDA (-3)     /* CUDA runtime / driver error (message has the CUDA error string) */
#define SOWB_ENOTSUP (-4)   /* device is not sm_100 */

#define SOWB_BF16 0
#define SOWB_F32 1
#define SOWB_F16 2   /* IEEE binary16 (torch.float16) */

enum sowb_op {
  SOWB_OP_LINEAR_FWD = 0,
  SOWB_OP_LINEAR_BWD = 1,
  SOWB_OP_MERGE = 2,
  SOWB_OP_THIN_QR = 3,
  SOWB_OP_TT_PROJECT = 4,
};

int sow_abi_version(void);
const char* sow_last_error(void);

/*
 * Live per-kernel timing for bench.py's roofline: while enabled, every launch of the classes below is bracketed
 * by CUDA events on the launching stream.  sow_profile_read sums elapsed milliseconds, algorithmic work (flops for
 * GEMM classes, bytes for merge / Adam) and the launch count of one class.  Classes: 0 forward GEMM (y), 1 dX GEMM,
 * 2 skinny GEMM (t_cat), 3 split-K GEMM (dA_cat), 4 grouped merge, 5 multi-tensor Adam, 6 fused dt + dB pass.
 */
int sow_profile_enable(int on);
int sow_profile_read(int klass, double* total_ms, double* total_work, int64_t* launches);

/* Rank padded to the k-block granularity used for the staged low-rank activations t / dt ([T, r_pad] bf16). */
int sow_rank_pad(int r);

/*
 * One projection of a GROUP of SoW linears that read the same input x[T,in] (q/k/v or gate/up of a transformer block;
 * a lone projection is a group of one).  All matrices row-major, of the call's dtype (the 2-byte tensors of SOWB_F32 are
 * bf16 pieces).  Members may differ in `out`, `r` and `scale`.
 */
typedef struct sowb_group_member {
  const void* W;    /* (in,out) frozen accumulation acc_downweight, or NULL before the first merge (sow.py:69-70) */
  const void* W_lo; /* SOWB_F32 mode: low bf16 piece of W (W ~ W + W_lo), else NULL                               */
  const void* A;    /* (in,r)   downscale_weights[i]                                                              */
  const void* B;    /* (r,out)  upscale_weights[i]                                                                */
  const void* bias; /* (out) or NULL                                              [forward]                      */
  void* y;          /* (T,out) output                                             [forward]                      */
  const void* dy;   /* (T,out) upstream gradient                                  [backward]                     */
  const void* dy_lo;/* SOWB_F32 mode: low bf16 piece of dY, else NULL             [backward]                     */
  void* dA;         /* (in,r)  gradient of A, or NULL                             [backward]                     */
  void* dB;         /* (r,out) gradient of B, or NULL                             [backward]                     */
  void* dbias;      /* (out)   gradient of bias, or NULL                          [backward]                     */
  int out, r;
  float scale;
} sowb_group_member;

/* Bytes of scratch sow_group_bwd needs (op = SOWB_OP_LINEAR_BWD; the forward needs none). */
size_t sow_group_workspace_bytes(int op, int64_t T, int in, const sowb_group_member* members_host, int n);

/*
 * Forward of a group.   Replaces SoWLinear.forward, tn_gradient/layer/sow.py:107-126, for every member i:
 *     y_i[T,out_i] = x[T,in] . W_i[in,out_i]  +  scale_i * (x . A_i[in,r_i]) . B_i[r_i,out_i]  (+ bias_i)
 * in 2 + n launches: the factors are packed into A_cat[in,R] = [A_0|0|A_1|0|...] (each member zero-padded to
 * sow_rank_pad(r_i) columns, R = their sum), ONE skinny GEMM computes t_cat[T,R] = scale_i * x . A_cat for all members
 * (x is read once instead of n times), and each y_i is one tcgen05 GEMM with the t_i . B_i product fused in as an extra
 * K-segment.  A_cat and t_cat (caller-allocated, bf16 in SOWB_BF16 / SOWB_F32, fp16 in SOWB_F16) are what autograd
 * saves for sow_group_bwd.
 * W_i may be NULL (pre-merge phase) -> rank-r term only.  1 <= n <= 4.
 *
 * dtype SOWB_BF16: everything bf16.  dtype SOWB_F16: everything fp16 (x, W, A, B, bias, y, A_cat, t_cat); x_lo and W_lo
 * must be NULL.  dtype SOWB_F32 (fp32 modules -- the reference's GLUE scripts never set a dtype,
 * run_glue.py:386-388,508-514): the fp32 operands arrive split into two bf16 pieces each (sow_split_bf16x2: v ~ hi + lo,
 * relative error 2^-17), x = (x, x_lo), W_i = (W, W_lo), and the base product runs as the bf16x3 contraction
 * x.W + x.W_lo + x_lo.W on the tensor cores with fp32 accumulation (fp32-faithful: ~1e-5 relative, vs 4e-3 for plain bf16
 * and 5e-4 for TF32); y_i and bias_i are fp32.  The rank-r factors A_i, B_i are passed rounded to bf16 (their products
 * are two orders of magnitude smaller than the base term).
 */
int sow_group_fwd(const void* x, const void* x_lo, const sowb_group_member* members_host, int n, void* A_cat, void* t_cat,
                  int64_t T, int in, int dtype, void* stream);

/* v (fp32, n elements) -> hi = bf16(v), lo = bf16(v - hi): the two pieces the SOWB_F32 mode consumes. */
int sow_split_bf16x2(const float* src, void* hi, void* lo, int64_t n, void* stream);

/*
 * Backward of a group.   Replaces the MmBackward nodes autograd records at sow.py:112,117,119 for every member:
 *     dt_i = scale_i * dY_i . B_i^T        dB_i = t_i^T . dY_i        (ONE pass over dY_i produces both)
 *     dA_cat = x^T . dt_cat                (ONE split-K GEMM for all members; x is read once)
 *     dX = sum_i dY_i . W_i^T + dt_cat . A_cat^T      (ONE GEMM with K-concatenated segments; NULL dx skips it)
 *     dbias_i = sum_T dY_i                 (if non-NULL)
 * The full in x out weight gradient is never formed (W is frozen: sow.py:69-70, prepare.py:142,150).  All reductions
 * across CTAs go through fp32 partials summed in a fixed order: results are bit-reproducible run to run.
 * dt_cat[T,R] (bf16, fp16 in SOWB_F16) is caller-allocated scratch.  At most 4 (SOWB_F32: 3) members may carry a dense W.
 * SOWB_F16: x, A_cat, t_cat, W, B, dY, dt_cat, dX, dA, dB and dbias are fp16; dy_lo and W_lo must be NULL.
 * SOWB_F32: dY_i = (dy, dy_lo) and W_i = (W, W_lo) are bf16 pieces, dX is fp32 (bf16x3 products); the factor gradients
 * are computed from the high pieces and written in bf16.
 */
int sow_group_bwd(const void* x, const void* A_cat, const void* t_cat, const sowb_group_member* members_host, int n,
                  void* dt_cat, void* dx, int64_t T, int in, int dtype, void* ws, size_t ws_bytes, void* stream);

/*
 * One entry of the grouped merge table (host memory, copied by the call).
 * Replaces SoWLinear.accumulate's dense branch, sow.py:131-134,140,151-153:  W <- W_prev + scale * A . B
 * W_prev may be NULL (first merge: W <- scale * A . B).  W and W_prev may alias (in-place RMW).
 */
typedef struct sowb_merge_entry {
  void* W;            /* (in,out) destination                     */
  const void* W_prev; /* (in,out) previous accumulation or NULL    */
  const void* A;      /* (in,r)                                    */
  const void* B;      /* (r,out)                                   */
  int in, out, r;
  float scale;
} sowb_merge_entry;

/* Grouped merge over n entries in ONE launch.  table_dev: device scratch of n * sow_merge_table_stride() bytes.
 * dtype SOWB_BF16: W, A, B bf16, the rank-r product on tcgen05, fp32 accumulate, one bf16 rounding of W per 64-wide
 *                  rank chunk.
 * dtype SOWB_F16 : the same with W, A, B fp16 and one fp16 rounding of W per rank chunk.
 * dtype SOWB_F32 : W, A, B fp32, exact fp32 FMA (fp32 modules keep their pretrained weights at full precision). */
size_t sow_merge_table_stride(void);
int sow_merge_grouped(const sowb_merge_entry* entries_host, int n, int dtype, void* table_dev,
                      size_t table_bytes, void* stream);

/*
 * Thin QR of the first r columns:  Q[m,r] (orthonormal) spanning X[:, :r] where X is (m,n) row-major fp32 with
 * leading dimension ldx.   Replaces the full-matrix torch.linalg.qr in qr_weight, tn_gradient/utils.py:19-22
 * (only Q[:, :rank] is kept: sow.py:171) and the complete QR in TensorTrain.decompose, tn_gradient/tt.py:129-132.
 * Batched: `batch` matrices, strides in elements.  Sign convention: R has non-negative diagonal.
 */
int sow_thin_qr(const float* X, int64_t x_batch_stride, int ldx, float* Q, int64_t q_batch_stride, int m, int r,
                int batch, void* ws /* sow_thin_qr_workspace_bytes(m, r, batch), 16-byte aligned */, size_t ws_bytes,
                void* stream);
/* scratch of sow_thin_qr: Cholesky factors, per-matrix flags and the fp64 Gram partials (summed in a fixed order: the
 * factorisation is bit-reproducible run to run) for r <= 64; batch*m*r*4 bytes for the Gram-Schmidt path above that. */
size_t sow_thin_qr_workspace_bytes(int m, int r, int batch);

/*
 * TT projection  R[r,n] = Q[m,r]^T . L[m,n]  in fp32 (3xTF32-free, exact fp32 FMA accumulate).
 * Replaces R[:right_rank,:] of the complete QR in tn_gradient/tt.py:129-133.  Batched like sow_thin_qr.
 */
int tt_project(const float* L, int64_t l_batch_stride, const float* Q, int64_t q_batch_stride, float* R,
               int64_t r_batch_stride, int m, int n, int r, int batch, void* ws, size_t ws_bytes, void* stream);
/* scratch of tt_project: when the m rows are split over CTAs each split stores a partial [r x n] and the partials are
 * summed in split order (bit-reproducible; no atomics).  0 when one split suffices (ws may then be NULL). */
size_t tt_project_workspace_bytes(int m, int n, int r, int batch);

/*
 * Fused pad + interleave for TensorTrain.from_matrix / from_tensor (tn_gradient/tt.py:48-67,33; utils.py:78-84),
 * any order d <= 8:   out[i1,o1,i2,o2,...,id,od] = src[(i1..id)_mm , (o1..od)_nn]   (0 outside (M,N))
 * src is (M,N) row-major of dtype `dtype`; out is fp32 with (mm*nn)^d elements.  tt_deinterleave is the inverse
 * restricted to (M,N) (TensorTrain.to_matrix, tt.py:242-247 + unpad_matrix, utils.py:86-87).
 */
int tt_interleave(const void* src, int M, int N, int mm, int nn, int order, float* out, int dtype, void* stream);
int tt_deinterleave(const float* src, int M, int N, int mm, int nn, int order, void* out, int dtype, void* stream);

/*
 * Order-2 TT of a matrix without materialising the padded + interleaved unfolding (tt.py:48-67 pads, reshapes and permutes:
 * three passes over M.N).  Element (ga, gb) of the P x P unfolding (P = mm*nn, ga = i1*nn + o1, gb = i2*nn + o2) is source
 * element (i1*mm + i2, o1*nn + o2), zero outside (M, N); the kernels address the source directly.
 *   tt_gather2      : X[P, ncols] = first ncols columns of the unfolding (input of sow_thin_qr)
 *   tt_project2     : R[r, P] = Q[P, r]^T . unfolding                     (TensorTrain.decompose, tt.py:129-133)
 *   tt_reconstruct2 : dst[M, N] = (G1[P, r] . G2[r, P]) de-interleaved and un-padded   (TensorTrain.to_matrix, tt.py:242-247)
 */
int tt_gather2(const void* src, int M, int N, int mm, int nn, float* X, int ncols, int dtype, void* stream);
int tt_project2(const void* src, int M, int N, int mm, int nn, const float* Q, float* R, int r, int dtype, void* ws,
                size_t ws_bytes, void* stream);
size_t tt_project2_workspace_bytes(int mm, int nn, int r);   /* split partials, as tt_project_workspace_bytes */
int tt_reconstruct2(const float* G1, const float* G2, int r, void* dst, int M, int N, int mm, int nn, int dtype, void* stream);

/* fp32 C[m,n] = A[m,r] . B[r,n] with small r: one link of the reconstruction chain (tt.py:213-237). */
int tt_matmul_rk(const float* A, const float* B, float* C, int m, int n, int r, void* stream);

/*
 * Order-2 TT reconstruction fused with the TT-Adam update.  Replaces, per parameter,
 * TensorTrain.reconstruct/to_matrix (tt.py:213-247) twice + the elementwise Adam of
 * tn_gradient/optimizer/ttadam.py:71-111:
 *     m = G1m . G2m ; v = max(G1v . G2v, 0)              (cores: G1 [(mm*nn), r], G2 [r, (mm*nn)], fp32)
 *     m = b1*m + (1-b1)*g ; v = b2*v + (1-b2)*g*g
 *     p -= step_size * m / (sqrt(v) + eps) ; p -= lr*wd*p  (if wd > 0)
 * and writes the NEW m, v in the padded+interleaved layout of tt_interleave (fp32, (mm*nn)^2 each) ready for
 * sow_thin_qr/tt_project, so the dense moments never round-trip HBM in (M,N) layout.
 * first_step != 0 -> previous m, v are zero (cores ignored; ttadam.py:68-70,76-78).
 */
int tt_adam_fused2(void* p, const void* g, const float* G1m, const float* G2m, const float* G1v,
                   const float* G2v, int r, float* m_out, float* v_out, int M, int N, int mm, int nn,
                   double beta1, double beta2, double eps, double step_size, double lr_wd, int first_step,
                   int dtype, void* stream);

/*
 * Order-2 TT-Adam with the re-compression fused in: the dense moments never reach HBM.  Same math as tt_adam_fused2
 * followed by sow_thin_qr + tt_project on its outputs, in three steps (ttadam.py:61-115):
 *   1. tt_adam2_head  : X{m,v}[P, 64] = the first 64 columns of the NEW moments (interleaved layout, P = mm*nn).
 *                       p is not modified.
 *   2. sow_thin_qr    : Q'{m,v}[P, r] from the first r columns of X{m,v}      (caller, batch = 2, ldx = 64)
 *   3. tt_adam2_fused : Adam update of p  +  R'{m,v}[r, P] = Q'^T . (new moments), accumulated tile by tile in
 *                       registers; each row range stores a partial in ws and the partials are summed in range order
 *                       (bit-reproducible; no atomics).  ws: tt_adam2_fused_workspace_bytes(mm, nn) bytes.
 * New cores: G1' = Q' (P x r), G2' = R' (r x P).  r <= 64.  first_step != 0 -> previous moments are zero.
 */
int tt_adam2_head(const void* g, const float* G1m, const float* G2m, const float* G1v, const float* G2v, int r, float* Xm,
                  float* Xv, int M, int N, int mm, int nn, double beta1, double beta2, int first_step, int dtype,
                  void* stream);
int tt_adam2_fused(void* p, const void* g, const float* G1m, const float* G2m, const float* G1v, const float* G2v, int r,
                   const float* Qm, const float* Qv, float* Rm, float* Rv, int M, int N, int mm, int nn, double beta1,
                   double beta2, double eps, double step_size, double lr_wd, int first_step, int dtype, void* ws,
                   size_t ws_bytes, void* stream);
size_t tt_adam2_fused_workspace_bytes(int mm, int nn);

/*
 * The whole order-2 TT-Adam step in one call, with both rank-r products on the tensor cores (tcgen05, operands split
 * into three bf16 pieces = fp32-accurate): tt_adam2_head -> sow_thin_qr -> operand split -> fused update + projection.
 * Outputs the new cores: Q'{m,v} (Qm, Qv = the two halves of one (2, P, r) array) and R'{m,v} (r x P each).
 * ws: tt_adam2_workspace_bytes(mm, nn) bytes, 256-byte aligned.  r <= 64.
 */
size_t tt_adam2_workspace_bytes(int mm, int nn);
int tt_adam2_step(void* p, const void* g, const float* G1m, const float* G2m, const float* G1v, const float* G2v, int r,
                  float* Qm, float* Qv, float* Rm, float* Rv, int M, int N, int mm, int nn, double beta1, double beta2,
                  double eps, double step_size, double lr_wd, int first_step, int dtype, void* ws, size_t ws_bytes,
                  void* stream);

/*
 * TT-Adam update for order > 2 on moments kept in the interleaved layout of tt_interleave ((mm*nn)^order fp32 elements each,
 * updated in place): the reconstruction chain already produces that layout and the decomposition sweep consumes it, so the
 * dense (M,N) moments of ttadam.py:71-84,113-115 never exist.  Padded positions are set to 0; v is clamped at 0 first.
 */
int tt_adam_interleaved(void* p, const void* g, float* m, float* v, int M, int N, int mm, int nn, int order, double beta1,
                        double beta2, double eps, double step_size, double lr_wd, int dtype, void* stream);

/*
 * The whole TT-Adam step of an order >= 3 tensor train in ONE call (TTAdam.step, ttadam.py:61-115, for "ranks" of length
 * order + 1 > 3): reconstruction chain of both moments into the interleaved layout (tt.py:213-237), the interleaved Adam
 * update of p (tt_adam_interleaved), and one decomposition sweep over both moments as a batch of two (tt.py:111-140).
 *   cores_in[k] / cores_out[k], k < order : the k-th core of BOTH moments, [2][r_k * P * r_{k+1}] fp32 (m first), P = mm*nn;
 *                                           cores_in may be NULL on the first step (zero moments).
 *   ranks[order + 1] with ranks[0] = ranks[order] = 1, inner ranks <= 64.
 * ws: tt_adam_nd_workspace_bytes(...) bytes (0 = unsupported shape), 256-byte aligned.
 */
size_t tt_adam_nd_workspace_bytes(int mm, int nn, int order, const int* ranks);
int tt_adam_nd_step(void* p, const void* g, const float* const* cores_in, float* const* cores_out, const int* ranks, int M, int N,
                  int mm, int nn, int order, double beta1, double beta2, double eps, double step_size, double lr_wd,
                  int first_step, int dtype, void* ws, size_t ws_bytes, void* stream);

/*
 * TensorTrain.from_matrix / to_matrix of an order >= 3 tensor train as ONE call each (tt.py:48-67,111-140 / 213-247):
 * tt_interleave + the thin-QR / projection sweep, and the reconstruction chain + tt_deinterleave.  cores[k]: the k-th core,
 * r_k * P * r_{k+1} fp32, P = mm*nn; ranks as in tt_adam_nd_step.  ws: tt_nd_workspace_bytes(...) (0 = unsupported), 256-byte
 * aligned.  src / dst: (M, N) row-major of dtype `dtype`.
 */
size_t tt_nd_workspace_bytes(int mm, int nn, int order, const int* ranks);
int tt_decompose_nd(const void* src, float* const* cores_out, const int* ranks, int M, int N, int mm, int nn, int order, int dtype,
                    void* ws, size_t ws_bytes, void* stream);
int tt_reconstruct_nd(const float* const* cores, const int* ranks, void* dst, int M, int N, int mm, int nn, int order, int dtype,
                      void* ws, size_t ws_bytes, void* stream);

/* Same update on dense fp32 moments m, v of shape (M,N) (no "ranks": the dense branch); v is clamped at 0 first (ttadam.py:84). */
int tt_adam_dense(void* p, const void* g, float* m, float* v, int64_t numel, double beta1, double beta2, double eps,
                  double step_size, double lr_wd, int dtype, void* stream);

/*
 * Multi-tensor Adam / AdamW: one launch over a device table of chunks
 *     struct { void* p; const void* g; void* m; void* v; int64_t n; }   (40 bytes, n <= sow_adam_chunk_elems())
 * covering all tensors of a param group (torch.optim.AdamW at scripts/simple_train.py:502-506).  Moments have
 * the parameter dtype (model.to(bf16): simple_train.py:425-426; torch.optim.AdamW keeps fp16 state for fp16 parameters
 * too); math is fp32 in registers.  dtype: SOWB_BF16, SOWB_F16 or SOWB_F32.  Bias corrections
 * are computed by the caller so `state["step"]` semantics (reset_optimizer, training_utils.py:257-277) stay on
 * the host side.  Hyper-parameters are doubles so that 1-beta is formed without float cancellation.
 * decoupled != 0 -> AdamW (p *= 1 - lr*wd), else L2 (g += wd*p).
 */
int sow_adam_chunk_elems(void);
int sow_adam_multi(const void* chunks_dev, int n_chunks, double lr, double beta1, double beta2, double eps,
                   double weight_decay, double bias_correction1, double bias_correction2, int decoupled, int dtype,
                   void* stream);
/* same, with the total element count of the table for the profiler's byte accounting */
int sow_adam_multi_ex(const void* chunks_dev, int n_chunks, int64_t total_elems, double lr, double beta1, double beta2,
                      double eps, double weight_decay, double bias_correction1, double bias_correction2, int decoupled,
                      int dtype, void* stream);

/*
 * CUDA-graph capturable variant: `step_dev` is a device fp32 counter that the call advances by one (a 1-thread kernel
 * ahead of the update) and from which the update kernel derives both bias corrections, so a captured optimizer step
 * replays correctly (torch.optim.AdamW(capturable=True) keeps state["step"] on the device for the same reason).
 */
int sow_adam_multi_dev(const void* chunks_dev, int n_chunks, int64_t total_elems, double lr, double beta1, double beta2,
                       double eps, double weight_decay, float* step_dev, int decoupled, int dtype, void* stream);

/*
 * Mixed-precision variant for loss-scaled training (torch.amp.GradScaler):
 *   state_dtype : dtype of m and v, either `dtype` or SOWB_F32 (fp32 moments for bf16 / fp16 parameters; each chunk-table
 *                 pointer is offset by its own tensor's element size).  p, g keep `dtype`.
 *   step_dev    : device step counter as in sow_adam_multi_dev, or NULL to use the host bias corrections (then both > 0).
 *   grad_scale  : device fp32 scalar or NULL.  g / *grad_scale (IEEE division) is the gradient of the update, and it is
 *                 written back into g, rounded to `dtype` (torch._fused_adamw_ does the same).
 *   found_inf   : device fp32 scalar or NULL; requires step_dev.  Non-zero: the update does nothing (p, m, v and g keep
 *                 every bit) and the step counter does not advance.
 * Arguments are validated (SOWB_EINVAL) before any work is queued or the CUDA context is touched.
 * Profiler bytes: (2 e_p + e_g + 4 e_state [+ e_g when grad_scale is given]) per element.
 */
int sow_adam_multi_amp(const void* chunks_dev, int n_chunks, int64_t total_elems, double lr, double beta1, double beta2,
                       double eps, double weight_decay, double bias_correction1, double bias_correction2, float* step_dev,
                       const float* grad_scale, const float* found_inf, int decoupled, int dtype, int state_dtype,
                       void* stream);

/*
 * Gradient clipping by the global 2-norm (torch.nn.utils.clip_grad_norm_, norm type 2), on the device and without atomics:
 *   sow_grad_norm_partials : one fp32 partial sum of squares per row of an Adam chunk table (reads g and n of each row;
 *                            dtype is the gradients' type), written to partials[0 .. n_chunks).  grad_scale: NULL, or
 *                            GradScaler's device scale, in which case each element is round_dtype(g / *grad_scale) -- the
 *                            value sow_adam_multi_amp's unscale writes back.  The tables of one param group write to
 *                            consecutive ranges of one partials buffer.
 *   sow_grad_norm_finalize : *total_norm = float(sqrt(sum of partials in fp64)), and the clip coefficient exactly as torch
 *                            computes it on an fp32 tensor: r = 1.0f / (total_norm + 1e-6f), c = r * (float)max_norm,
 *                            *clip_coef = min(c, 1) with NaN propagated.  An inf norm gives 0, a NaN norm NaN.
 *   sow_adam_multi_clip    : sow_adam_multi_amp with the gradient round(round(g / scale) * *clip_coef) (the unscale only when
 *                            grad_scale is given), which is also written back into g.  found_inf still skips everything.
 * Every result is bit-reproducible.  Arguments are validated (SOWB_EINVAL) before any work is queued or the CUDA context
 * is touched: unknown dtypes, n_chunks < 0, NULL pointers where a value is needed, n_partials < 1, max_norm not finite or
 * not > 0, and the dtype combinations sow_adam_multi_amp rejects.
 */
int sow_grad_norm_partials(const void* chunks_dev, int n_chunks, int dtype, const float* grad_scale, float* partials,
                           void* stream);
int sow_grad_norm_finalize(const float* partials, int n_partials, double max_norm, float* total_norm, float* clip_coef,
                           void* stream);
int sow_adam_multi_clip(const void* chunks_dev, int n_chunks, int64_t total_elems, double lr, double beta1, double beta2,
                        double eps, double weight_decay, double bias_correction1, double bias_correction2, float* step_dev,
                        const float* grad_scale, const float* found_inf, const float* clip_coef, int decoupled, int dtype,
                        int state_dtype, void* stream);

/*
 * Element-wise glue of the Llama block (HF transformers modeling_llama.py), bit-identical to the eager chains it replaces.
 * dtype SOWB_BF16 or SOWB_F16; math in fp32, each result rounded to the 16-bit type where eager rounds (see glue.cu).
 * Pointers 16-byte aligned.  One launch per call.
 *
 * Rotary embedding of q and k (apply_rotary_pos_emb):  out = q * cos + rotate_half(q) * sin, the same for k.
 *   q: (B, Hq, S, D) with element strides q_sb, q_sh, q_ss and a contiguous last dimension; k: (B, Hk, S, D) likewise.
 *   cos, sin: (B or 1, S, D) contiguous; cs_sb is their batch stride (0 when shared by the batch).
 *   q_out, k_out: (B, S, H, D) contiguous -- the layout of eager's q_embed seen through its (B, H, S, D) transpose.
 *   D a multiple of 16, strides multiples of 8.
 * sow_rope_bwd: dq, dk of the same layout from the upstream gradients gq, gk (strided like q, k); cos / sin as above.
 */
int sow_rope_fwd(const void* q, const void* k, const void* cos, const void* sin, void* q_out, void* k_out, int B, int S, int Hq,
                 int Hk, int D, int64_t q_sb, int64_t q_sh, int64_t q_ss, int64_t k_sb, int64_t k_sh, int64_t k_ss,
                 int64_t cs_sb, int dtype, void* stream);
int sow_rope_bwd(const void* gq, const void* gk, const void* cos, const void* sin, void* dq, void* dk, int B, int S, int Hq,
                 int Hk, int D, int64_t gq_sb, int64_t gq_sh, int64_t gq_ss, int64_t gk_sb, int64_t gk_sh, int64_t gk_ss,
                 int64_t cs_sb, int dtype, void* stream);

/*
 * SwiGLU gate of LlamaMLP (act_fn = silu) over n contiguous elements:
 *   sow_swiglu_fwd: h = silu(gate) * up
 *   sow_swiglu_bwd: dup = dh * silu(gate),  dgate = silu_backward(dh * up, gate)   (one pass over dh, gate, up)
 */
int sow_swiglu_fwd(const void* gate, const void* up, void* h, int64_t n, int dtype, void* stream);
int sow_swiglu_bwd(const void* dh, const void* gate, const void* up, void* dgate, void* dup, int64_t n, int dtype,
                   void* stream);

/*
 * LlamaRMSNorm over rows x width contiguous elements, bit-identical to the eager HF forward and its autograd backward:
 *   sow_rmsnorm_fwd: rs = rsqrt(mean(x^2) + eps) per row (fp32, rows values), y = w * (x * rs)
 *   sow_rmsnorm_bwd: dx from dy, x, w and the saved rs; when p is not null also p = dy * (x * rs), the per-element
 *                    product whose sum over the rows is dw.
 * width one of 128, 256, 512, 768, 1024, 2048, 3072, 4096; rows >= 16 unless width == 128 (torch's row sums take
 * another order below that); x, w, y, dy, dx, p 16-byte aligned.  rows == 0 does nothing.
 */
int sow_rmsnorm_fwd(const void* x, const void* w, void* y, float* rs, int64_t rows, int width, float eps, int dtype,
                    void* stream);
int sow_rmsnorm_bwd(const void* dy, const void* x, const void* w, const float* rs, void* dx, void* p, int64_t rows,
                    int width, int dtype, void* stream);

/*
 * Cross-entropy of rows x vocab contiguous 16-bit logits against int64 targets, bit-identical to torch's fp32
 * log_softmax of the upcast logits and the backward of log_softmax + the upcast:
 *   sow_ce_fwd: per row, fp32 row_max = max_j x_j, row_logsum = log(sum_j exp(x_j - row_max)) and
 *               logp_t = (x_t - row_max) - row_logsum; logp_t = 0 for a target outside [0, vocab), whose row is not gathered
 *   sow_ce_bwd: grad = d(sum_i dlogp_t[i] * logp_t[i]) / d logits (16-bit, the logits' shape) from the forward's row_max
 *               and row_logsum; dlogp_t[i] is the NLL gradient of row i (0 for an ignored row)
 * vocab a multiple of 8 in [16384, 32768] (torch's log_softmax reduces other widths in another order); logits and grad
 * 16-byte aligned.  rows == 0 does nothing.
 */
int sow_ce_fwd(const void* logits, const int64_t* target, float* row_max, float* row_logsum, float* logp_t, int64_t rows,
               int vocab, int dtype, void* stream);
int sow_ce_bwd(const void* logits, const float* row_max, const float* row_logsum, const int64_t* target,
               const float* dlogp_t, void* grad, int64_t rows, int vocab, int dtype, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SOW_B200_H_ */

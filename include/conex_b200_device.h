/* conex-b200 device layer — the thin C ABI between the C++ host orchestration
 * (conex_b200/csrc/host) and the hand-written sm_100a CUDA kernels (conex_b200/csrc/device).
 *
 * Conventions
 *  - every pointer named d_* / marked "device" is a plain device pointer (cudaMalloc'ed by the
 *    caller, e.g. torch.Tensor.data_ptr()); no torch or CUDA types appear in the signatures;
 *  - `stream` is a cudaStream_t passed as void* (NULL = default stream);
 *  - matrices are column-major FP64 with an explicit leading dimension;
 *  - every call returns 0 on success, a cudaError_t value (>0) if a launch failed, or -1 for bad
 *    arguments. Kernels are asynchronous on `stream`; results that the host needs are written to
 *    device memory and fetched by the caller.
 *
 * Each entry point names the reference code whose arithmetic it replaces (SURVEY.md §8a).
 */
#ifndef CONEX_B200_DEVICE_H
#define CONEX_B200_DEVICE_H
#include <stddef.h>
#ifdef __cplusplus
extern "C" {
#endif

/* ---- K1/K2/K3/K7/K8 workhorse: FP64 tensor-core (DMMA.8x8x4) GEMM --------------------------
 * C[b] = alpha * op(A[b]) * op(B[b]) + beta * C[b],  b = 0..batch-1 (strided batches).
 * op(A) is M x K, op(B) is K x N. lower_only != 0 computes/stores only tiles and entries with
 * row >= col (SYRK-style Gram and Cholesky trailing updates).
 * Replaces Eigen GEMM at dense_lmi_constraint.cc:31-32,77-78, psd_constraint.cc:25,61,79,
 * exponential_map_pade.cc:13-17, block_triangular_operations.cc:205-216. */
int cxb_dgemm(void* stream, int transA, int transB, int M, int N, int K, double alpha,
              const double* dA, long lda, long strideA, const double* dB, long ldb, long strideB,
              double beta, double* dC, long ldc, long strideC, int batch, int lower_only);

/* Same with explicit control, used by the tuning harness (tools/gemm_tune.py) and the Schur assembly:
 * config = tile configuration (-1: chosen from the shape), splits = split-K factor (0: automatic,
 * deterministic fixed-order reduction), mirror != 0 (needs lower_only, M == N) also stores
 * C[col,row] so that the result is exactly symmetric; diag_off shifts the lower_only test to
 * row + diag_off >= col (a row panel starting diag_off rows below the top of a lower-triangular
 * result). */
int cxb_dgemm_ex(void* stream, int config, int splits, int transA, int transB, int M, int N, int K,
                 double alpha, const double* dA, long lda, long strideA, const double* dB, long ldb,
                 long strideB, double beta, double* dC, long ldc, long strideC, int batch,
                 int lower_only, int mirror, int diag_off);
/* Tile configuration used for large shapes when config < 0 (process-wide; tuning only). */
/* A/B arm: C = A B (plain NN, strided batch; tri = 1: B lower triangular) with the operand tiles staged by the TMA
 * engine's bulk copies (cp.async.bulk + mbarrier) into the same padded shared-memory layout; bit-identical results.
 * Needs K % 16 == 0, even M / leading dimensions / strides, 16-byte aligned operands; returns -1 otherwise. */
int cxb_dgemm_bulk(void* stream, int M, int N, int K, const double* dA, long lda, long strideA, const double* dB,
                   long ldb, long strideB, double* dC, long ldc, long strideC, int batch, int tri);
void cxb_set_default_gemm_config(int config);
/* Tile configuration of the deep A^T B contractions (Gram matrices of the Schur assembly): -1 (default) = the default
 * configuration of the other large products; 6 = 64 x 128 tiles with 32 x 64 warp tiles. A/B switch. */
void cxb_set_gram_gemm_config(int config);
/* Deterministic split-K policy of deep contractions: 0 (default) = split only to fill the machine; k > 0 = additionally
 * cap the k-tiles (of 16) one CTA walks at k, so that CTAs sharing operand panels stay within L2 of each other. */
void cxb_set_gemm_split_policy(int max_ktiles_per_cta);

/* ---- K1+K2: Schur complement of one dense LMI block -----------------------------------------
 * dAall: (m+1) contiguous column-major n x n matrices: A_0..A_{m-1} followed by C.
 * dW: n x n scaling point. dB: scratch of (m+2)*n*n doubles (receives W A_i W, W C W, W).
 * dT: scratch of panel*n*n doubles (panel >= 1 constraint matrices scaled per pass).
 * dHaug: (m+2) x (m+1) column-major, ld = ldh >= m+2. On return (lower trapezoid):
 *   Haug[i][j] = tr(W A_i W A_j) (i >= j, i,j < m)        -> H  (dense_lmi_constraint.cc:72-78)
 *   Haug[m][j] = <W C W, A_j> = AQc_j ; Haug[m][m] = <c,Qc>   (:80, :84-88)
 *   Haug[m+1][j] = <W, A_j> = AW_j  ; Haug[m+1][m] = <w,c>     (:79, :82)
 */
int cxb_schur_dense_lmi(void* stream, int n, int m, const double* dAall, const double* dW,
                        double* dB, double* dT, int panel, double* dHaug, long ldh);

/* Same Newton system through the symmetric form: with W = L L^T, H_ij = <L^T A_i L, L^T A_j L>. The
 * scaled matrices are formed with triangular-aware DMMA GEMMs (zero k-tiles skipped) and stored as
 * packed lower 64 x 64 tiles, then one SYRK-shaped Gram (K = 0.54 n^2) gives Haug. Executes
 * 1.33 m n^3 + 0.54 m^2 n^2 flop instead of 3 m n^3 + m^2 n^2 (reference: 4 m n^3 + m^2 n^2,
 * dense_lmi_constraint.cc:62-103). dX: (m + 2) * cxb_packed_symmetric_size(n) doubles, dT: panel * n * n,
 * dL: n * n (receives the Cholesky factor of W). d_info[0] != 0 on return means W was not numerically
 * positive definite: Haug is then invalid and the caller must use cxb_schur_dense_lmi. */
size_t cxb_packed_symmetric_size(int n);
int cxb_pack_symmetric(void* stream, int n, const double* d_src, double* d_dst);
int cxb_schur_dense_lmi_sym(void* stream, int n, int m, const double* dAall, const double* dW, double* dX,
                            double* dT, int panel, double* dL, int* d_info, double* dHaug, long ldh);
/* The two phases of cxb_schur_dense_lmi_sym on their own: K1 (factor W, scale and pack every matrix, the packed
 * identity in row m + 1 of X) and K2 (the Gram of the packed rows). */
int cxb_schur_dense_lmi_sym_scale(void* stream, int n, int m, const double* dAall, const double* dW, double* dX,
                                  double* dT, int panel, double* dL, int* d_info);
int cxb_schur_dense_lmi_sym_gram(void* stream, int n, int m, const double* dX, double* dHaug, long ldh);

/* ---- entry-sparse LMI operators (MaxCut, Lovasz theta, ...; sparse_lmi.cu) -----------------------
 * A_i given by their non-zero entries (both triangles listed): entries offsets[i] .. offsets[i+1]-1 of
 * rows / cols / vals. Same Haug as cxb_schur_dense_lmi, from O((sum nnz)^2) gathers out of W instead
 * of matrix products. dC: dense n x n affine term. d_work: 2 n*n doubles (C W, W C W). */
int cxb_sparse_lmi_schur(void* stream, int n, int m, const int* d_offsets, const int* d_rows,
                         const int* d_cols, const double* d_vals, const double* dC, const double* dW,
                         double* d_work, double* dHaug, long ldh);
/* out = sum_i y_i A_i - k C with the entries grouped by matrix position (column-major index):
 * position t holds entries pos_ptr[t] .. pos_ptr[t+1]-1 of (pos_var, pos_val); fixed summation order. */
int cxb_sparse_lmi_slack(void* stream, int n, int npos, const int* d_pos_ptr, const long* d_pos_index,
                         const int* d_pos_var, const double* d_pos_val, const double* dC, const double* dy,
                         double k, double* d_out);

/* Same result with bounded scratch: dBp holds (panel + 1) * n * n doubles (one row panel of scaled
 * matrices, contracted immediately), dT panel * n * n. Used when a second A-sized buffer does not fit. */
int cxb_schur_dense_lmi_streamed(void* stream, int n, int m, const double* dAall, const double* dW,
                                 double* dBp, double* dT, int panel, double* dHaug, long ldh);

/* ---- K3: blocked right-looking Cholesky, lower, in place (block_triangular_operations.cc:184-219,
 * Eigen::LLT). d_info (device int) is set to 0 on success or to (1 + index of the first
 * non-positive pivot). d_work: at least cxb_potrf_worksize(m) doubles. */
size_t cxb_potrf_worksize(int m);
int cxb_potrf_lower(void* stream, int m, double* dH, long ldh, double* d_work, int* d_info);
/* The same factorisation step by step, for the multi-GPU driver (host/distributed_cholesky.cc):
 * cxb_potrf_begin clears d_info; cxb_potrf_panel factors the block column [j0, j0 + w) x rows
 * [j0, m) in place (w <= cxb_potrf_max_panel(); the columns must already carry the updates of all
 * block columns to their left) and is a no-op once d_info != 0; the trailing updates are
 * cxb_dgemm(..., lower_only = 1) calls issued by the caller. */
int cxb_potrf_max_panel(void);
int cxb_potrf_begin(void* stream, int* d_info);
int cxb_potrf_panel(void* stream, int m, int j0, int w, double* dH, long ldh, int* d_info);

/* ---- K3/K5 by supernodes (reference block_triangular_operations.cc:184-219 per supernode, :114-182
 * for the solves; host/supernodal_kkt_solver.cc drives them front by front):
 * cxb_potrf_partial factors the first `cols` columns of a rows x cols lower trapezoid (L11 on top,
 * L21 = A21 L11^{-T} below) without resetting d_info; cxb_trsv_lower is one substitution sweep with a
 * triangular block; cxb_scatter_lower_indexed adds sign * (lower triangle of an n x n matrix) into
 * arbitrary destinations (d_idx: one offset per pair a >= b in column-major order of the lower
 * triangle, negative = skip) — the assembly of a cone's G and the Schur update of a separator
 * (supernodal_assembler.cc:103-165, block_triangular_operations.cc:205-216); cxb_front_forward /
 * cxb_front_backward apply a front's L21 to the separator entries of the right-hand side. */
int cxb_potrf_partial(void* stream, int rows, int cols, double* dF, long ld, int* d_info);
int cxb_trsv_lower(void* stream, int m, const double* dL, long ldl, double* dx, int transposed);
int cxb_scatter_lower_indexed(void* stream, int n, const double* dG, long ldg, const long* d_idx, double sign,
                              double* d_dst);
int cxb_front_forward(void* stream, int p, int sk, const double* dL21, long ld, const double* d_xk,
                      const int* d_sep, double* d_x);
int cxb_front_backward(void* stream, int p, int sk, const double* dL21, long ld, double* d_xk,
                       const int* d_sep, const double* d_x);

/* ---- K5: triangular solves with the Cholesky factor (block_triangular_operations.cc:114-182):
 * X <- L^{-T} L^{-1} X for nrhs right-hand sides (columns of dX, leading dimension ldx). */
int cxb_potrs_lower(void* stream, int m, const double* dL, long ldl, double* dX, long ldx, int nrhs);

/* ---- K4: diagonally pivoted, regularised LDL^T (block_triangular_operations.cc:315-349 +
 * Eigen::RLDLT, RLDLT.h:297-431) for KKT systems with equality constraints.
 * The reference picks pivots by the largest *stored* diagonal entry of a left-looking algorithm,
 * i.e. by the ORIGINAL diagonal, so the whole permutation is known before any arithmetic: the host
 * computes it from diag(K) (host/cone_program.cc), cxb_sym_permute_lower forms P K P^T from the
 * lower triangle, and cxb_ldlt_lower factors it WITHOUT further pivoting as L S L^T, S = diag(+-1)
 * (LDL^T with |D|^{1/2} folded into L) by a blocked right-looking algorithm: 128-column diagonal
 * blocks in shared memory, panel solve, DMMA trailing update. Pivots with |d| <= 1e-9 become
 * +-1e-9 (RLDLT.h:378-389); d_info[1] = 1 then (regularization_used), d_info[0] stays 0.
 * d_signs: N doubles (S). d_work: cxb_ldlt_worksize(N) doubles. */
size_t cxb_ldlt_worksize(int N);
int cxb_sym_permute_lower(void* stream, int N, const double* dK, long ldk, const int* d_perm,
                          double* dKp, long ldp);
int cxb_ldlt_lower(void* stream, int N, double* dK, long ldk, double* d_signs, double* d_work,
                   int* d_info);
/* x <- P^T L^{-T} S L^{-1} P x (block_triangular_operations.cc:222-312); perm[i] = original index
 * at pivot position i; d_tmp: N doubles. */
int cxb_ldlt_solve(void* stream, int N, const double* dL, long ldl, const double* d_signs,
                   const int* d_perm, double* dx, double* d_tmp);
/* ---- LDL^T over the fronts of the multifrontal solver (reference BlockLDLTInPlace,
 * block_triangular_operations.cc:315-349: Eigen::RLDLT of every supernode's diagonal block, pivoting inside it) ----
 * cxb_front_permute: dOut <- the front dF (rows x s lower trapezoid) under the supernode's pivot order: diagonal
 *   block P F11 P^T, separator block with permuted columns.
 * cxb_ldlt_partial: signed factorisation of the first `cols` columns of a rows x cols trapezoid: on top L11 with
 *   F11 = L11 S L11^T, below G = F21 L11^{-T} S; the Schur complement of the rows below is F22 - G S G^T.
 *   d_work: rows * 128 doubles. d_info[1] (regularised pivots, RLDLT.h:378-389) is reset by cxb_ldlt_begin only.
 * cxb_scale_columns: dOut[:, c] = dA[:, c] * d_signs[c]   (G S for that Schur complement).
 * cxb_permute_vec / cxb_apply_signs: the per-supernode permutations and S of the solves. */
int cxb_ldlt_begin(void* stream, int* d_info);
int cxb_front_permute(void* stream, int rows, int s_cols, const double* dF, long ld, const int* d_perm, double* dOut,
                      long ldo);
int cxb_ldlt_partial(void* stream, int rows, int cols, double* dF, long ld, double* d_signs, double* d_work,
                     int* d_info);
int cxb_scale_columns(void* stream, int rows, int cols, const double* dA, long lda, const double* d_signs,
                      double* dOut, long ldo);
int cxb_permute_vec(void* stream, int N, const int* d_perm, const double* d_in, double* d_out, int scatter);
int cxb_apply_signs(void* stream, int N, const double* d_signs, double* dx);

/* ---- K6: negative slack  out = sum_j coef[j] * Aall[:, j]  (dense_lmi_constraint.cc:8-27);
 * Aall is nn x cols column-major (ld = nn), d_coef has `cols` entries (y followed by -k for C). */
int cxb_gemv_n(void* stream, long nn, int cols, const double* dAall, const double* d_coef,
               double* d_out);

/* ---- K7: two-sided Lanczos (approximate_eigenvalues.cc:178-239) ------------------------------
 * d_WS, d_W: n x n (ld n; W symmetric). Start vector: d_r (n entries) when d_col_index is NULL,
 * otherwise column (int)*d_col_index of the n x n matrix d_r (the index stays on the device, so no
 * host round trip is needed after the diag-argmax reduction). Runs at most num_iter steps with the reference's
 * breakdown test (beta^2 < 1e-6). Outputs: d_alpha[num_iter], d_beta[num_iter], d_count[0] = number
 * of valid beta entries (alpha has d_count+1 valid entries). d_work: cxb_lanczos_worksize(n)
 * doubles. d_count: 2 ints (see cxb_lanczos_two_sided_range). */
size_t cxb_lanczos_worksize(int n);
int cxb_lanczos_two_sided(void* stream, int n, const double* d_WS, const double* d_W,
                          const double* d_r, const double* d_col_index, int num_iter,
                          double* d_alpha, double* d_beta, int* d_count, double* d_work);

/* Same with the breakdown rule of the incremental (Hermitian) LMI: rel_tol > 0 stops when
 * beta^2 < rel_tol * <U, U> of the first step (jordan_matrix_algebra.cc:421-433, rel_tol = 1e-5);
 * rel_tol == 0 is cxb_lanczos_two_sided. */
int cxb_lanczos_two_sided_ex(void* stream, int n, const double* d_WS, const double* d_W,
                             const double* d_r, const double* d_col_index, int num_iter,
                             double* d_alpha, double* d_beta, int* d_count, double* d_work,
                             double rel_tol);

/* Steps j_begin .. j_end-1 only (j_begin == 0 also runs the set-up). d_count has TWO ints:
 * d_count[0] as above, d_count[1] = 1 once the recurrence has stopped (breakdown or num_iter
 * reached), so a caller can run a short first range, look, and skip the rest. */
int cxb_lanczos_two_sided_range(void* stream, int n, const double* d_WS, const double* d_W,
                                const double* d_r, const double* d_col_index, int num_iter, int j_begin,
                                int j_end, double* d_alpha, double* d_beta, int* d_count, double* d_work,
                                double rel_tol);

/* ---- K7 reductions (psd_constraint.cc:63-80,107-127). d_out slots (all device doubles):
 *   out[0] = tr(WS), out[1] = sum_ij WS_ij WS_ji = tr(WS WS), out[2] = argmax_i WS_ii (as double),
 *   out[3] = max_i WS_ii. */
int cxb_ws_reductions(void* stream, int n, const double* d_WS, double* d_out);

/* ---- K8: geodesic update  W <- sym( pade33( scale * (WS + e_weight I) ) W )
 * (psd_constraint.cc:13-28, exponential_map_pade.cc:10-32). d_WS is destroyed.
 * d_work: cxb_geodesic_worksize(n) doubles; d_iwork: 2n ints (pivots + permutation). d_info: device int, 0 or
 * 1 + index of a zero pivot. */
size_t cxb_geodesic_worksize(int n);
int cxb_geodesic_update(void* stream, int n, double* d_W, double* d_WS, double e_weight,
                        double scale, double* d_work, int* d_iwork, int* d_info);

/* K9 exponential: d_out = (I + X/4 + X^2/32)^4 (DoExponentialMap<1>, exponential_map.cc:15-42);
 * d_work: n*n doubles. And the geodesic update built on it (hermitian_psd.cc:9-31); d_work: 2 n*n. */
int cxb_taylor_expm(void* stream, int n, const double* d_X, double* d_out, double* d_work);
int cxb_geodesic_update_taylor(void* stream, int n, double* d_W, double* d_WS, double e_weight,
                               double scale, double* d_work);

/* Padé map alone: d_out = pade33(d_X) (exponential_map_pade.cc:23-32). d_X is preserved. */
int cxb_pade_expm(void* stream, int n, const double* d_X, double* d_out, double* d_work,
                  int* d_iwork, int* d_info);

/* Partial-pivot LU solve A X = B (A n x n destroyed, B n x nrhs overwritten by X). */
int cxb_lu_solve(void* stream, int n, double* dA, long lda, int nrhs, double* dB, long ldb,
                 int* d_ipiv, int* d_info);

/* ---- small vector / matrix helpers used by the host loop -------------------------------------*/
/* W <- I (psd_constraint.cc:92-95) */
int cxb_set_identity(void* stream, int n, double* dW);
/* out[0] = x . y  (n entries) */
int cxb_dot(void* stream, long n, const double* dx, const double* dy, double* d_out);
/* y <- a*x + b*y + c*z (z may be NULL) */
int cxb_axpbypcz(void* stream, long n, double a, const double* dx, double b, double* dy, double c,
                 const double* dz);
/* strided copy: dst[i*incd] = src[i*incs] */
int cxb_copy_strided(void* stream, long n, const double* src, long incs, double* dst, long incd);
/* H[idx[a], idx[b]] (+)= G[a, b] for a >= b (lower) — supernodal_assembler.cc:103-165 in dense form */
int cxb_scatter_add_lower(void* stream, int mc, const double* dG, long ldg, const int* d_idx,
                          double* dH, long ldh);
/* dst[0..n) = value */
int cxb_fill(void* stream, long n, double value, double* d_dst);
/* dst[idx[i]] += src[i] / dst[i] = src[idx[i]]  (idx NULL = identity) — the clique gather/scatter of
 * constraint_manager.h:107-124 and cone_program.h:59-67 */
int cxb_scatter_add_vec(void* stream, int n, const double* d_src, const int* d_idx, double* d_dst);
int cxb_gather_vec(void* stream, int n, const double* d_src, const int* d_idx, double* d_dst);
/* out = K x, K symmetric N x N given by its lower triangle — the residual of the iterative refinement
 * (kkt_solver.cc:248-261) */
int cxb_symv_lower(void* stream, int N, const double* dK, long ld, const double* dx, double* d_out);
/* W <- (1 + w_e) W + WSW  (psd_constraint.cc:33-43) */
int cxb_affine_update(void* stream, int n, double* dW, const double* dWSW, double w_e);

/* ---- small cones, batched: one CTA per program of a batch (small_cones.cu) --------------------
 * The LP cone (conex/linear_constraint.cc), the second-order cone (conex/soc_constraint.cc) and
 * small dense LMI blocks (n*n doubles fit in shared memory; conex/psd_constraint.cc +
 * dense_lmi_constraint.cc) of `batch` structurally identical programs, advanced in lock step; the
 * single-program LP / SOC plugins are the batch == 1 case. Problem p of the batch uses
 * ptr + p * stride of every array below.
 *   data : rows x (m + 1) column-major, rows = n (LP), n + 1 (SOC), n * n (PSD); columns 0..m-1 hold
 *          the linear operator (PSD: vec(A_j)), column m the affine term.
 *   state: LP  W[n] t1[n] t2[n] at offsets 0, np, 2 np (np = n rounded up to 4)
 *          SOC (W0, W1)[n + 1] at 0, d[n + 1] at op (op = n + 1 rounded up to 4)
 *          PSD W, T1, T2 (n x n each) at 0, nnp, 2 nnp (nnp = n * n rounded up to 4)
 *   work : SOC (n + 1) * (m + 4) doubles; PSD (m + 2) * n * n doubles; LP none.
 *   y_offset: where the cone's y starts in the slack kernels' y argument (cxb_small_eigen / cxb_small_prepare and their
 *          _multi forms): program p reads y[p * ystride + y_offset + j], j < m. 0 for a cone on all variables; a cone
 *          on a subset of a program's variables reads the slice that cxb_small_gather placed behind the program's y.
 *          It fills the padding after `m`, so the size and layout of the struct are those of earlier releases, and
 *          a zero-initialised descriptor reads y from its start.
 * active (device ints, may be NULL) masks programs that must not be touched. */
enum { CXB_CONE_LP = 0, CXB_CONE_SOC = 1, CXB_CONE_PSD = 2 };
typedef struct {
  int type, n, m;
  int y_offset;
  const double* data;
  long data_stride;
  double* state;
  long state_stride;
  double* work;
  long work_stride;
  /* optional, PSD only: the lower triangles of the m + 1 matrices, column by column, n (n + 1) / 2 doubles each
   * (cxb_small_pack_symmetric); when not NULL the slack kernels (cxb_small_eigen / cxb_small_prepare) read it instead of
   * the full matrices — half the HBM traffic of the two passes a Newton step makes over the operator for its slacks. */
  const double* packed;
  long packed_stride;
} cxb_small_cone;
size_t cxb_small_state_size(int type, int n);
size_t cxb_small_work_size(int type, int n, int m);
int cxb_small_set_identity(void* stream, int batch, const cxb_small_cone* cone, const int* d_active);
/* Packed copy of a PSD cone's operator: d_packed[p * packed_stride + j * kp + c n - c (c - 1) / 2 + (r - c)] = A_j[r, c],
 * r >= c, kp = n (n + 1) / 2. *d_asymmetric (device int, zeroed by the caller) is set when some A_j[r, c] != A_j[c, r]:
 * the packed copy then does not represent the operator and must not be used (the reference forms the slack from the
 * full matrices, dense_lmi_constraint.cc:8-20). */
int cxb_small_pack_symmetric(void* stream, int batch, const cxb_small_cone* cone, double* d_packed, long packed_stride,
                             int* d_asymmetric);
/* The same for the matrices [first, first + count) of the m + 1 only (0 <= first, 1 <= count, first + count <= m + 1):
 * refreshes the packed copy after an in-place update of those columns of `data`; the other matrices are neither read
 * nor written. cxb_small_pack_symmetric is the full range. */
int cxb_small_pack_symmetric_columns(void* stream, int batch, const cxb_small_cone* cone, int first, int count,
                                     double* d_packed, long packed_stride, int* d_asymmetric);
/* G (ldg, lower triangle), AW, AQc (m each, stride vstride), scal[2] = {<w,c>, <c,Qc>} (stride
 * sstride): assigned (accumulate == 0) or added to (ConstructSchurComplementSystem, initialize flag). */
int cxb_small_schur(void* stream, int batch, const cxb_small_cone* cone, double* dG, long ldg,
                    long gstride, double* dAW, double* dAQc, long vstride, double* d_scal,
                    long sstride, int accumulate, const int* d_active);
/* A/B switch of the dense-LMI branch of cxb_small_schur for blocks of order n <= 32, n % 4 == 0
 * (device/small_psd_mma.cuh): 2 (default) = DMMA kernel, one slot per warp, two CTAs per SM; 1 = DMMA kernel with the
 * whole operator of a program in shared memory, one CTA per SM; 0 = the DFMA team kernel. */
void cxb_set_small_psd_mma(int enabled);
/* Thread layout of the other small-cone kernels: 2 (default) = one WARP per program for the triangular solves of the
 * small KKT systems (several programs per CTA, __syncwarp + shuffles), one CTA of 128 threads per program for the
 * kernels with parallel phases; 1 = warp layout everywhere; 0 = CTA layout everywhere. Same arithmetic. */
void cxb_set_small_team_mode(int mode);
/* out4 = {lambda_min, lambda_max, frobenius_norm_squared, trace} of Q(w^{1/2})(c_weight c - A y)
 * (GetWeightedSlackEigenvalues). c_weight: per-program device array d_cw (stride 1) when not NULL,
 * else the scalar. */
int cxb_small_eigen(void* stream, int batch, const cxb_small_cone* cone, const double* dy, long ystride,
                    double c_weight, const double* d_cw, double* d_out4, long ostride,
                    const int* d_active);
/* out2 = {norminfd, normsqrd} (PrepareStep); affine != 0: the dual-recovery update. */
int cxb_small_prepare(void* stream, int batch, const cxb_small_cone* cone, const double* dy,
                      long ystride, int affine, double c_weight, const double* d_cw, double e_weight,
                      double* d_out2, long ostride, const int* d_active);
/* TakeStep with step size `step` (or d_step[p]); d_info[p] != 0 reports a singular Padé system. */
int cxb_small_take_step(void* stream, int batch, const cxb_small_cone* cone, double step,
                        const double* d_step, double e_weight, int* d_info, const int* d_active);
/* The four per-cone operations on `ncones` cones of every program in ONE launch (grid = programs x cones; up to 8
 * cones per launch, longer lists are chunked): the lock step of a batch of multi-cone programs (reference
 * cone_program.cc:173-214, :416-436 loop over the constraints) otherwise serialises the cones' dependent chains.
 * Cone k writes d_out + 4 k (+ p * ostride). Same arithmetic as the per-cone calls, bit for bit. */
int cxb_small_set_identity_multi(void* stream, int batch, int ncones, const cxb_small_cone* cones,
                                 const int* d_active);
int cxb_small_eigen_multi(void* stream, int batch, int ncones, const cxb_small_cone* cones, const double* dy,
                          long ystride, double c_weight, const double* d_cw, double* d_out4, long ostride,
                          const int* d_active);
int cxb_small_prepare_multi(void* stream, int batch, int ncones, const cxb_small_cone* cones, const double* dy,
                            long ystride, int affine, double c_weight, const double* d_cw, double e_weight,
                            double* d_out2, long ostride, const int* d_active);
int cxb_small_take_step_multi(void* stream, int batch, int ncones, const cxb_small_cone* cones, double step,
                              const double* d_step, double e_weight, int* d_info, const int* d_active);
/* CTA size (32, 64 or 128 threads; default 64) of cxb_small_eigen / cxb_small_prepare in the CTA layout: their
 * phases are short dependent chains, so what bounds them is the number of cones resident per SM. */
void cxb_set_small_cone_threads(int threads);
/* A/B switch: 0 = the *_multi entry points launch their cones one after the other (default 1). */
void cxb_set_small_fused_launches(int enabled);
/* Cones on variable subsets in a batch: the gather of their y slices and the scatter-add of their Schur blocks.
 * cxb_small_gather: y[p * ystride + dst + i] = y[p * ystride + d_idx[i]] for i < count with d_idx[i] >= 0 (entries
 * < 0 are padding and leave their slot alone). Every d_idx[i] must be < dst: the sources, a program's variables,
 * lie before the destination slices. One CTA per program. */
int cxb_small_gather(void* stream, int batch, int count, const int* d_idx, double* dy, long ystride, long dst,
                     const int* d_active);
/* The batched counterpart of cxb_scatter_add_lower + cxb_scatter_add_vec: for the subset cones k < ncones in order,
 * d_cones[3 k ..] = {m_k, first, offset}: the cone's variables are d_idx[first .. first + m_k), and its Schur
 * block (cxb_small_schur with accumulate = 0) lies at dS + p * sstride + offset as G_k (m_k x m_k lower triangle,
 * ld = m_k rounded up to 4), then AW_k and AQc_k (ld doubles each), then its two scalars. Adds G_k[i, j], i >= j,
 * to H[max(v_i, v_j), min(v_i, v_j)], AW_k / AQc_k to AW / AQc at v, the scalars to scal[0..1]. accumulate == 0
 * first zeroes the leading m x m block of H, AW[0..m), AQc[0..m) and scal[0..1]. One CTA per program; the cones
 * are added one after the other (no atomics: the result does not depend on scheduling). */
int cxb_small_scatter_schur(void* stream, int batch, int ncones, const int* d_cones, const int* d_idx, const double* dS,
                            long sstride, int m, double* dH, long ldh, long hstride, double* dAW, double* dAQc,
                            long vstride, double* d_scal, long scal_stride, int accumulate, const int* d_active);
/* Cholesky of `batch` N x N matrices (lower, ld, stride) and solves with nrhs = 1; d_info[p] = 0 or
 * 1 + first column whose pivot is not > 0, in column order (a NaN pivot fails too; block_triangular_operations.cc:
 * 184-219, :114-182). After a failure the contents of that program's H are unspecified. d_active[p] == 0 masks
 * programs that must not be touched. Any N whose matrices fit in device memory: up to N = 170 the whole matrix of a
 * program is factored in shared memory; above that cxb_small_potrf_blocked is used. */
int cxb_small_potrf(void* stream, int batch, int N, double* dH, long ldh, long hstride, int* d_info,
                    const int* d_active);
/* The same contract at any N, blocked: block columns of 32, the diagonal block in shared memory, the trailing update
 * on the FP64 tensor cores, the matrix factored in place in global memory; shared memory per program does not
 * depend on N. Not bitwise equal to the shared-memory kernel (the summation order differs). */
int cxb_small_potrf_blocked(void* stream, int batch, int N, double* dH, long ldh, long hstride, int* d_info,
                            const int* d_active);
int cxb_small_potrs(void* stream, int batch, int N, const double* dL, long ldl, long lstride, double* dX,
                    long xstride, const int* d_active);
/* Regularised LDL^T of `batch` symmetric indefinite N x N matrices (KKT systems with equality multipliers; the
 * batched counterpart of cxb_sym_permute_lower + cxb_ldlt_lower, one program per CTA like cxb_small_potrf): per
 * program the pivot order of Eigen::RLDLT from diag(K) (RLDLT.h:328-356, as CONEXB200_RldltPivotOrder), the
 * permuted copy P K P^T gathered from the lower triangle of K, and its factorisation L S L^T, S = diag(+-1), with
 * |D|^{1/2} folded into L. Pivots with |d| <= 1e-9 become -1e-9 when d < 0, +1e-9 otherwise; d_info[p] = 1 then,
 * else 0 — it never fails. K is not modified; the lower triangle of L (ldl, lstride), d_perm (ints, perm[i] =
 * original index at pivot position i) and d_signs (S) are written. d_active[p] == 0 masks programs that must not be
 * touched. Any N whose matrices fit in device memory: up to N = 169 the permuted copy (N^2 + O(N) doubles) is
 * factored in shared memory; above that cxb_small_ldlt_blocked is used. */
int cxb_small_ldlt(void* stream, int batch, int N, const double* dK, long ldk, long kstride, double* dL, long ldl,
                   long lstride, int* d_perm, long pstride, double* d_signs, long sstride, int* d_info,
                   const int* d_active);
/* The same contract at any N, blocked like cxb_small_potrf_blocked: P K P^T is gathered straight into L, which is
 * then factored in place; shared memory per program: a fixed amount plus the pivot order (N doubles, N ints). */
int cxb_small_ldlt_blocked(void* stream, int batch, int N, const double* dK, long ldk, long kstride, double* dL,
                           long ldl, long lstride, int* d_perm, long pstride, double* d_signs, long sstride,
                           int* d_info, const int* d_active);
/* x <- P^T L^{-T} S L^{-1} P x with the factors of cxb_small_ldlt, nrhs = 1. */
int cxb_small_ldlt_solve(void* stream, int batch, int N, const double* dL, long ldl, long lstride, const int* d_perm,
                         long pstride, const double* d_signs, long sstride, double* dX, long xstride,
                         const int* d_active);
/* out[p] = a[p] x[p] + b[p] y[p] + c[p] z[p] (n entries each; coefficient arrays on the device,
 * NULL coefficient array / vector = term absent). */
int cxb_batched_lincomb(void* stream, int batch, int n, const double* d_a, const double* dx, long xs,
                        const double* d_b, const double* dy, long ys, const double* d_c,
                        const double* dz, long zs, double* d_out, long os, const int* d_active);
/* out[p * ostride] = x[p] . y[p] */
int cxb_batched_dot(void* stream, int batch, int n, const double* dx, long xs, const double* dy, long ys,
                    double* d_out, long ostride);

#ifdef __cplusplus
}
#endif
#endif

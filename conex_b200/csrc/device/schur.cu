// K1 + K2: Schur-complement assembly for one dense LMI block, H_ij = tr(A_i W A_j W), on the tensor
// cores (FP64, and for the symmetric form's Gram the 8-bit integer ones, see below).
//
// Reference (dense_lmi_constraint.cc:62-103): per constraint two n x n x n GEMMs (A_i W, W A_i W)
// followed by a GEMV against the growing slab Avect[:, 0:i+1] — BLAS-2 and memory bound. Here:
//   K1  T_i = A_i W          one strided-batched DMMA GEMM per panel of constraints
//       B_i = W T_i          strided-batched, lower tiles only + mirrored store (B_i symmetric)
//   K2  Haug = Bmat^T Aall   one lower-trapezoid DMMA GEMM with K = n^2 (SYRK-style Gram)
// The affine term C rides along as matrix m of Aall and W as row m+1 of Bmat, so the same Gram
// launch also yields AQc_j = <W C W, A_j>, AW_j = <W, A_j>, <c,Qc> and <w,c> (rows m, m+1 of Haug).
#include "common.cuh"
#include "device_api.h"

namespace cxb {
namespace {

// dst (packed 64 x 64 lower tiles, off-diagonal tiles scaled by sqrt 2) <- symmetric src (n x n)
__global__ void PackSymmetricKernel(int n, const double* __restrict__ src, double* dst) {
  const int T = (n + 63) / 64;
  const int tn = blockIdx.y, tm = blockIdx.x;
  if (tm < tn) return;
  const long slot = (long)tn * T - (long)tn * (tn - 1) / 2 + (tm - tn);
  const double sc = (tm == tn) ? 1.0 : 1.4142135623730951;
  for (int e = threadIdx.x; e < 4096; e += blockDim.x) {
    const int rl = e & 63, cl = e >> 6;
    const int r = tm * 64 + rl, c = tn * 64 + cl;
    dst[slot * 4096 + e] = (r < n && c < n) ? sc * src[(long)c * n + r] : 0.0;
  }
}

// L <- lower triangle of W, strict upper triangle zeroed (the triangular GEMMs read stored zeros
// inside the diagonal tiles)
__global__ void CopyLowerKernel(int n, const double* __restrict__ W, double* L) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  const int c = blockIdx.y;
  if (r >= n) return;
  L[(long)c * n + r] = (r >= c) ? W[(long)c * n + r] : 0.0;
}

}  // namespace
}  // namespace cxb

// ---- symmetric form -----------------------------------------------------------------------------------
// With W = L L^T:  H_ij = tr(A_i W A_j W) = <L^T A_i L, L^T A_j L>, so the Schur complement is the Gram
// matrix of the scaled matrices S_i = L^T A_i L ("form W^{1/2} A_i W^{1/2}, then a SYRK-style Gram").
// K1 forms S_i in n^3 flops, as LAPACK's dsygst does, from A_i = V_i + V_i^T with V_i = tril(A_i, -1) + diag(A_i) / 2:
//   K1  Y_i = V_i L            lower x lower = lower: lower tiles only, into dT             (n^3 / 3 flop)
//       S_i = L^T Y_i + Y_i^T L  symmetric: lower tiles only, both products in one k loop (2 n^3 / 3 flop)
//           stored as packed 64 x 64 lower tiles with sqrt(2)-scaled off-diagonal tiles, so that the
//           plain dot product of two packed matrices is their trace inner product (K = 0.54 n^2)
//   K2  Haug = X^T X (lower)   X = [S_0 .. S_{m-1}, L^T C L, I]: one SYRK-shaped Gram, emulated on the 8-bit integer
//                              tensor cores (ozaki.cu) at sizes where that pays, one DMMA GEMM below them
// K1 reads the lower triangle of A_i and C only. Rows m and m+1 of Haug are AQc_j = <L^T C L, S_j> and
// AW_j = tr(S_j) as before. Executed flops: 1.0 m n^3 + 0.54 m^2 n^2 against 3 m n^3 + m^2 n^2 of the W A_i W form
// (4 m n^3 + m^2 n^2 dense).
// dL: n*n scratch for the factor; d_info[0] != 0 reports a W that is not numerically positive definite
// (the caller then falls back to cxb_schur_dense_lmi). dX: (m + 2) * cxb_packed_symmetric_size(n).
extern "C" size_t cxb_packed_symmetric_size(int n) { return (size_t)cxb::PackedSymmetricSize(n); }

extern "C" int cxb_pack_symmetric(void* stream, int n, const double* d_src, double* d_dst) {
  using namespace cxb;
  const int T = (n + 63) / 64;
  CountLaunch(); PackSymmetricKernel<<<dim3(T, T), 256, 0, AsStream(stream)>>>(n, d_src, d_dst);
  return LaunchStatus();
}

// The two phases are separate entry points so that the sharded assembly can start shipping its scaled matrices to
// the peers as soon as K1 is done, under its own Gram.
extern "C" int cxb_schur_dense_lmi_sym_scale(void* stream, int n, int m, const double* dAall, const double* dW,
                                             double* dX, double* dT, int panel, double* dL, int* d_info) {
  using namespace cxb;
  cudaStream_t s = AsStream(stream);
  if (n < 1 || m < 1 || panel < 1) return -1;
  const long nn = (long)n * n;
  const long kp = PackedSymmetricSize(n);
  CountLaunch(); CopyLowerKernel<<<dim3((n + 127) / 128, n), 128, 0, s>>>(n, dW, dL);
  int rc = cxb_potrf_lower(stream, n, dL, n, nullptr, d_info);
  if (rc) return rc;
  const int total = m + 1;  // A_0..A_{m-1}, C
  for (int p0 = 0; p0 < total; p0 += panel) {
    const int pb = (panel < total - p0) ? panel : (total - p0);
    rc = DgemmStructured(s, -1, 1, false, false, n, n, n, 1.0, dAall + (long)p0 * nn, n, nn, dL, n, 0, 0.0, dT,
                         n, nn, pb, true, false, 0, kHalfLowerTimesLower, false);
    if (rc) return rc;
    rc = DgemmStructured(s, -1, 1, true, false, n, n, n, 1.0, dL, n, 0, dT, n, nn, 0.0, dX + (long)p0 * kp, n,
                         kp, pb, true, false, 0, kSyr2kLower, /*pack=*/true);
    if (rc) return rc;
  }
  // row m + 1 of the Gram: the packed identity, AW_j = tr(S_j) = <I, S_j>
  rc = SetIdentity(s, n, dT);
  if (rc) return rc;
  return cxb_pack_symmetric(stream, n, dT, dX + (long)(m + 1) * kp);
}

// K2 runs on the 8-bit integer tensor cores (FP64 emulation, ozaki.cu) when there are at least two 128-row tile rows and
// one full 2^15 K chunk, and on the DMMA Gram otherwise (a handful of CTAs, where slicing X costs as much as the
// product). _ws: dWork holds cxb_schur_dense_lmi_sym_gram_workspace(n, m) bytes for the slices of X, or is nullptr (the
// caller could not afford them: DMMA Gram). Without the argument the slices come from the stream-ordered pool for the
// call, and the DMMA Gram runs if that allocation fails.
extern "C" size_t cxb_schur_dense_lmi_sym_gram_workspace(int n, int m) {
  const long kp = cxb::PackedSymmetricSize(n);
  return (m + 2 >= 256 && kp >= (1L << 15)) ? cxb::GramEmulatedWorkspace(m + 2, kp) : 0;
}

extern "C" int cxb_schur_dense_lmi_sym_gram_ws(void* stream, int n, int m, const double* dX, double* dHaug, long ldh,
                                               void* dWork, size_t work_bytes) {
  using namespace cxb;
  if (n < 1 || m < 1 || ldh < m + 2) return -1;
  cudaStream_t s = AsStream(stream);
  const long kp = PackedSymmetricSize(n);
  const size_t need = cxb_schur_dense_lmi_sym_gram_workspace(n, m);
  if (need > 0 && dWork != nullptr && work_bytes >= need) {
    return GramEmulated(s, m + 2, m + 1, kp, dX, kp, dHaug, ldh, dWork);
  }
  return Dgemm(s, true, false, m + 2, m + 1, (int)kp, 1.0, dX, kp, 0, dX, kp, 0, 0.0, dHaug, ldh, 0, 1, true);
}

extern "C" int cxb_schur_dense_lmi_sym_gram(void* stream, int n, int m, const double* dX, double* dHaug, long ldh) {
  const size_t need = cxb_schur_dense_lmi_sym_gram_workspace(n, m);
  void* p = nullptr;
  if (need > 0 && cudaMallocAsync(&p, need, cxb::AsStream(stream)) != cudaSuccess) {
    cudaGetLastError();
    p = nullptr;
  }
  const int rc = cxb_schur_dense_lmi_sym_gram_ws(stream, n, m, dX, dHaug, ldh, p, need);
  if (p != nullptr) cudaFreeAsync(p, cxb::AsStream(stream));
  return rc;
}

extern "C" int cxb_schur_dense_lmi_sym(void* stream, int n, int m, const double* dAall, const double* dW,
                                       double* dX, double* dT, int panel, double* dL, int* d_info,
                                       double* dHaug, long ldh) {
  if (ldh < m + 2) return -1;
  const int rc = cxb_schur_dense_lmi_sym_scale(stream, n, m, dAall, dW, dX, dT, panel, dL, d_info);
  if (rc) return rc;
  return cxb_schur_dense_lmi_sym_gram(stream, n, m, dX, dHaug, ldh);
}

extern "C" int cxb_schur_dense_lmi(void* stream, int n, int m, const double* dAall, const double* dW,
                                   double* dB, double* dT, int panel, double* dHaug, long ldh) {
  using namespace cxb;
  cudaStream_t s = AsStream(stream);
  if (n < 1 || m < 1 || panel < 1 || ldh < m + 2) return -1;
  const long nn = (long)n * n;
  const int total = m + 1;  // A_0..A_{m-1}, C
  for (int p0 = 0; p0 < total; p0 += panel) {
    const int pb = (panel < total - p0) ? panel : (total - p0);
    int rc = Dgemm(s, false, false, n, n, n, 1.0, dAall + (long)p0 * nn, n, nn, dW, n, 0, 0.0, dT, n,
                   nn, pb, false);
    if (rc) return rc;
    // B_i = W T_i is symmetric in exact arithmetic: compute the lower tiles only and mirror them
    // (3 n^3 instead of 4 n^3 flops per constraint, and B_i exactly symmetric).
    rc = DgemmEx(s, -1, 1, false, false, n, n, n, 1.0, dW, n, 0, dT, n, nn, 0.0, dB + (long)p0 * nn, n,
                 nn, pb, true, true);
    if (rc) return rc;
  }
  cudaMemcpyAsync(dB + (long)(m + 1) * nn, dW, sizeof(double) * nn, cudaMemcpyDeviceToDevice, s);
  return Dgemm(s, true, false, m + 2, m + 1, (int)nn, 1.0, dB, nn, 0, dAall, nn, 0, 0.0, dHaug, ldh, 0,
               1, true);
}

// Same result without ever materialising all of B: one row panel of scaled matrices at a time is
// formed and immediately contracted against the constraint matrices to its left
// (Haug[p0 + q, c] = <B_q, A_c>, c <= p0 + q). dBp: (panel + 1) * n * n doubles, dT: panel * n * n.
// Memory: A + two panels instead of 2 A — what lets config 5 (n = 1000, m = 20000, A = 160 GB) run on
// one 192 GB B200. Cost: A is re-read once per row panel ((m / panel) / 2 passes over A in total).
extern "C" int cxb_schur_dense_lmi_streamed(void* stream, int n, int m, const double* dAall,
                                            const double* dW, double* dBp, double* dT, int panel,
                                            double* dHaug, long ldh) {
  using namespace cxb;
  cudaStream_t s = AsStream(stream);
  if (n < 1 || m < 1 || panel < 1 || ldh < m + 2) return -1;
  const long nn = (long)n * n;
  const int total = m + 1;  // A_0..A_{m-1}, C
  for (int p0 = 0; p0 < total; p0 += panel) {
    const int pb = (panel < total - p0) ? panel : (total - p0);
    int rc = Dgemm(s, false, false, n, n, n, 1.0, dAall + (long)p0 * nn, n, nn, dW, n, 0, 0.0, dT, n,
                   nn, pb, false);
    if (rc) return rc;
    rc = DgemmEx(s, -1, 1, false, false, n, n, n, 1.0, dW, n, 0, dT, n, nn, 0.0, dBp, n, nn, pb, true,
                 true);
    if (rc) return rc;
    int rows = pb;
    if (p0 + pb == total) {  // last panel: W rides along as row m + 1 (AW_j = <W, A_j>, <w,c>)
      cudaMemcpyAsync(dBp + (long)pb * nn, dW, sizeof(double) * nn, cudaMemcpyDeviceToDevice, s);
      rows = pb + 1;
    }
    const int cols = (p0 + rows < total) ? (p0 + rows) : total;
    rc = DgemmEx(s, -1, 0, true, false, rows, cols, (int)nn, 1.0, dBp, nn, 0, dAall, nn, 0, 0.0,
                 dHaug + p0, ldh, 0, 1, true, false, p0);
    if (rc) return rc;
  }
  return LaunchStatus();
}

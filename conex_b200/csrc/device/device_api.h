// Internal C++ view of the device layer (namespace cxb). The extern "C" surface that the host
// orchestration and the tests bind is include/conex_b200_device.h.
#pragma once
#include <cuda_runtime.h>

#include "../../../include/conex_b200_device.h"

namespace cxb {

// gemm.cu
int Dgemm(cudaStream_t stream, bool transA, bool transB, int M, int N, int K, double alpha,
          const double* A, long lda, long sA, const double* B, long ldb, long sB, double beta,
          double* C, long ldc, long sC, int batch, bool lower_only);
// Full-control variant: config < 0 = pick from the shape, splits == 0 = automatic split-K,
// mirror = also store the transposed entries of a lower_only square result; with lower_only the
// entries kept are those with row + diag_off >= col (row panels of a lower-triangular result).
int DgemmEx(cudaStream_t stream, int config, int splits, bool transA, bool transB, int M, int N, int K,
            double alpha, const double* A, long lda, long sA, const double* B, long ldb, long sB,
            double beta, double* C, long ldc, long sC, int batch, bool lower_only, bool mirror,
            int diag_off = 0);

// What a structured GEMM knows about its operands (square, lower_only results; k-tiles inside the zero parts
// are skipped, stored zeros cover the rest; always the 64 x 64 x 16 tile of configuration 2, no split-K):
enum GemmStructure : int {
  kGeneral = 0,
  // C = alpha S B (A, B untransposed, beta = 0), S = tril(A, -1) + diag(A) / 2, B lower triangular with stored zeros
  // above its diagonal. Only the lower triangle of A is ever part of the result (entries above it are selected
  // away, not multiplied), so A may hold anything there. C is lower triangular; its diagonal tiles are stored
  // whole, the strict upper part as exact zeros.
  kHalfLowerTimesLower = 1,
  // C = alpha (A^T B + B^T A) (transA, B untransposed, lda == ldb), A and B lower triangular with stored zeros
  // above their diagonals inside the diagonal tiles; the diagonal tiles of C are computed whole.
  kSyr2kLower = 2,
};

// Structured variant: see GemmStructure; pack = the (square, lower_only) result is written as packed 64 x 64
// lower tiles, PackedSymmetricSize(n) doubles per matrix (stride sC), off-diagonal tiles scaled by
// sqrt(2) so that the plain dot product of two packed symmetric matrices is their trace inner product.
int DgemmStructured(cudaStream_t stream, int config, int splits, bool transA, bool transB, int M, int N,
                    int K, double alpha, const double* A, long lda, long sA, const double* B, long ldb,
                    long sB, double beta, double* C, long ldc, long sC, int batch, bool lower_only,
                    bool mirror, int diag_off, GemmStructure structure, bool pack);
long PackedSymmetricSize(int n);

// cholesky.cu: factors the block column [j0, j0 + w) x rows [j0, m) in place (w <= 512)
int PotrfBlockColumn(cudaStream_t s, int m, int j0, int w, double* H, long ldh, int* info);

// blas1.cu
int SetIdentity(cudaStream_t s, int n, double* W);
int Symmetrize(cudaStream_t s, int n, double* W);                          // W <- (W + W^T)/2
int ShiftScale(cudaStream_t s, int n, double* X, double e, double scale);  // X <- scale (X + e I)
int ScaleAddDiag(cudaStream_t s, int n, const double* X, double a, double d, double* Y);  // Y = aX + dI
int SumDiff(cudaStream_t s, long total, const double* U, const double* V, double* N, double* D);
int Transpose(cudaStream_t s, int n, const double* X, double* XT);

// lu.cu
int LuFactor(cudaStream_t s, int n, double* A, long lda, int* ipiv, int* info);
int LuSolveFactored(cudaStream_t s, int n, const double* LU, long lda, const int* ipiv, int nrhs,
                    double* B, long ldb, double* tmp, int* perm);
int PadeExpm(cudaStream_t s, int n, const double* X, double* out, double* work, int* iwork, int* info);

}  // namespace cxb

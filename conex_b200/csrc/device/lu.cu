// K8: geodesic update of the PSD scaling point — [3/3] Padé matrix exponential as a GEMM chain on
// the FP64 tensor cores plus a blocked partial-pivot LU solve.
//
// Replaces PsdConstraint::GeodesicUpdate (psd_constraint.cc:13-28) and
// ExponentialMapPadeApproximation / ComputeWeightedPowers (exponential_map_pade.cc:10-32):
//   X  = scale * (WS + e I);  X2 = X X;  U = X (X2 + 60 I);  V = 12 X2 + 120 I
//   E  = (V - U)^{-1} (V + U)   (partial pivoting, like Eigen partialPivLu)
//   W <- sym(E W)
// There is deliberately no scaling-and-squaring: the reference relies on the step-size rule to
// keep ||X|| small, and adding it would change the iterates.
#include "common.cuh"
#include "device_api.h"

namespace cxb {
namespace {

constexpr int kLuNB = 32;      // LU panel width
constexpr int kSolveNB = 128;  // block size of the multi-RHS triangular solves
constexpr int kRhsCols = 32;   // RHS columns per CTA in the diagonal-block solves

// Factor the panel A[j0:n, j0:j0+nb] with row pivoting. One CTA of 1024 threads working in
// global memory (the panel is L2 resident). Row swaps are applied inside the panel only.
__global__ void __launch_bounds__(1024) LuPanelKernel(int n, int j0, int nb, double* A, long ld,
                                                      int* ipiv, int* info) {
  __shared__ double s_val[32];
  __shared__ int s_idx[32];
  __shared__ double s_row[kLuNB];
  __shared__ int s_piv;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int j = 0; j < nb; j++) {
    const int col = j0 + j;
    double* Ac = A + (long)col * ld;
    // 1. pivot search
    double best = -1.0;
    int arg = col;
    for (int r = col + tid; r < n; r += 1024) {
      const double v = fabs(Ac[r]);
      if (v > best) {
        best = v;
        arg = r;
      }
    }
    for (int o = 16; o > 0; o >>= 1) {
      const double ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
      if (ob > best || (ob == best && oa < arg)) {
        best = ob;
        arg = oa;
      }
    }
    if (lane == 0) {
      s_val[warp] = best;
      s_idx[warp] = arg;
    }
    __syncthreads();
    if (tid == 0) {
      double b = s_val[0];
      int a = s_idx[0];
      for (int w = 1; w < 32; w++) {
        if (s_val[w] > b || (s_val[w] == b && s_idx[w] < a)) {
          b = s_val[w];
          a = s_idx[w];
        }
      }
      s_piv = a;
      ipiv[col] = a;
      if (b == 0.0 && *info == 0) *info = col + 1;
    }
    __syncthreads();
    const int p = s_piv;
    // 2. swap rows col <-> p inside the panel, and stage the pivot row
    if (tid < nb) {
      double* c = A + (long)(j0 + tid) * ld;
      const double a = c[col], b = c[p];
      if (p != col) {
        c[col] = b;
        c[p] = a;
      }
      s_row[tid] = b;  // new A[col, j0 + tid]
    }
    __syncthreads();
    const double piv = s_row[j];
    const double inv = (piv != 0.0) ? 1.0 / piv : 0.0;
    // 3. multipliers + rank-1 update of the remaining panel columns
    for (int r = col + 1 + tid; r < n; r += 1024) {
      const double l = Ac[r] * inv;
      Ac[r] = l;
      for (int c = j + 1; c < nb; c++) A[(long)(j0 + c) * ld + r] -= l * s_row[c];
    }
    __syncthreads();
  }
}

// The same panel factorisation with the active columns in shared memory: the panel is processed in
// sub-panels of SW columns (SW * rows * 8 B of shared memory, rows = n - j0), each factored column by
// column entirely on chip (pivot search, swap, rank-1 update: three barriers and no global traffic
// per column), then written back and applied to the panel's remaining columns (unit-lower solve of
// their SW pivot rows + one rank-SW update in global memory). The kernel above pays the L2 round
// trips of a rank-1 update of up to 31 columns after every column: 211 us per 2000 x 32 panel, 46 %
// of the whole geodesic update (profiles/r01_g_geodesic_n2000_launches.txt).
template <int SW>
__global__ void __launch_bounds__(1024) LuPanelSmemKernel(int n, int j0, int nb, double* A, long ld,
                                                          int* ipiv, int* info) {
  extern __shared__ double sm[];  // sm[c * rows + r]: column j0 + q0 + c, row j0 + r
  __shared__ double s_val[32];
  __shared__ int s_idx[32];
  __shared__ double s_prow[SW];        // pivot row of the sub-panel
  __shared__ double s_u[SW][kLuNB];    // solved pivot rows of the remaining panel columns
  __shared__ int s_piv;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int rows = n - j0;
  // Row interchanges of the panel columns that are not on chip are split-phase: the two loads are
  // issued in the swap phase of column j and consumed (stored crosswise) in the swap phase of column
  // j + 1, so that their L2 latency hides behind the rank-1 update and the next pivot search instead
  // of stalling the barrier. Same thread, same column: program order keeps overlapping swaps exact.
  double* const gcol = A + (long)(j0 + (tid < nb ? tid : 0)) * ld + j0;
  double held_a = 0, held_b = 0;
  int held_col = 0, held_p = 0;
  bool held = false;
  for (int q0 = 0; q0 < nb; q0 += SW) {
    const int sw = min(SW, nb - q0);
    for (int c = 0; c < sw; c++) {
      const double* Ac = A + (long)(j0 + q0 + c) * ld + j0;
      for (int r = q0 + tid; r < rows; r += 1024) sm[c * rows + r] = Ac[r];
    }
    __syncthreads();
    for (int j = 0; j < sw; j++) {
      const int col = q0 + j;  // panel-local pivot position
      const double* sc = sm + j * rows;
      // 1. pivot search: largest |a|, smallest row on ties
      double best = -1.0;
      int arg = col;
      for (int r = col + tid; r < rows; r += 1024) {
        const double v = fabs(sc[r]);
        if (v > best) {
          best = v;
          arg = r;
        }
      }
      for (int o = 16; o > 0; o >>= 1) {
        const double ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
        if (ob > best || (ob == best && oa < arg)) {
          best = ob;
          arg = oa;
        }
      }
      if (lane == 0) {
        s_val[warp] = best;
        s_idx[warp] = arg;
      }
      __syncthreads();
      if (warp == 0) {
        best = s_val[lane];
        arg = s_idx[lane];
        for (int o = 16; o > 0; o >>= 1) {
          const double ob = __shfl_xor_sync(0xffffffffu, best, o);
          const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
          if (ob > best || (ob == best && oa < arg)) {
            best = ob;
            arg = oa;
          }
        }
        if (lane == 0) {
          s_piv = arg;
          ipiv[j0 + col] = j0 + arg;
          if (best == 0.0 && *info == 0) *info = j0 + col + 1;
        }
      }
      __syncthreads();
      const int p = s_piv;
      // 2. swap rows col <-> p over the whole panel (sub-panel columns on chip, the others in global)
      if (tid < nb) {
        const int c = tid - q0;
        if (c >= 0 && c < sw) {
          const double a = sm[c * rows + col], b = sm[c * rows + p];
          sm[c * rows + col] = b;
          sm[c * rows + p] = a;
          s_prow[c] = b;
        } else {
          if (held) {
            gcol[held_col] = held_b;
            gcol[held_p] = held_a;
            held = false;
          }
          if (p != col) {
            held_a = gcol[col];
            held_b = gcol[p];
            held_col = col;
            held_p = p;
            held = true;
          }
        }
      }
      __syncthreads();
      const double piv = s_prow[j];
      const double inv = (piv != 0.0) ? 1.0 / piv : 0.0;
      // 3. multipliers + rank-1 update of the sub-panel's remaining columns
      for (int r = col + 1 + tid; r < rows; r += 1024) {
        const double l = sm[j * rows + r] * inv;
        sm[j * rows + r] = l;
#pragma unroll
        for (int c = 1; c < SW; c++) {
          if (j + c < sw) sm[(j + c) * rows + r] -= l * s_prow[j + c];
        }
      }
      __syncthreads();
    }
    if (held) {  // complete the last interchange before anyone reads these columns
      gcol[held_col] = held_b;
      gcol[held_p] = held_a;
      held = false;
    }
    // write the factored sub-panel back
    for (int c = 0; c < sw; c++) {
      double* Ac = A + (long)(j0 + q0 + c) * ld + j0;
      for (int r = q0 + tid; r < rows; r += 1024) Ac[r] = sm[c * rows + r];
    }
    __syncthreads();
    const int rem = nb - q0 - sw;
    if (rem > 0) {
      // pivot rows of the remaining columns: u <- L11^{-1} u (unit lower, sw x sw), one thread per column
      if (tid < rem) {
        double* g = A + (long)(j0 + q0 + sw + tid) * ld + j0 + q0;
        double u[SW];
#pragma unroll
        for (int k = 0; k < SW; k++) u[k] = (k < sw) ? g[k] : 0.0;
#pragma unroll
        for (int k = 1; k < SW; k++) {
#pragma unroll
          for (int kk = 0; kk < k; kk++) {
            if (k < sw) u[k] -= sm[kk * rows + q0 + k] * u[kk];
          }
        }
#pragma unroll
        for (int k = 0; k < SW; k++) {
          if (k < sw) g[k] = u[k];
          s_u[k][tid] = u[k];
        }
      }
      __syncthreads();
      // rows below: A[r, c] -= sum_k L[r, q0 + k] U[q0 + k, c]
      for (int r = q0 + sw + tid; r < rows; r += 1024) {
        double l[SW];
#pragma unroll
        for (int k = 0; k < SW; k++) l[k] = (k < sw) ? sm[k * rows + r] : 0.0;
        double* g = A + (long)(j0 + q0 + sw) * ld + j0 + r;
        for (int c0 = 0; c0 < rem; c0 += 8) {
          double a[8];
#pragma unroll
          for (int c = 0; c < 8; c++) a[c] = (c0 + c < rem) ? g[(long)(c0 + c) * ld] : 0.0;
#pragma unroll
          for (int c = 0; c < 8; c++) {
#pragma unroll
            for (int k = 0; k < SW; k++) a[c] -= l[k] * s_u[k][(c0 + c) & (kLuNB - 1)];
          }
#pragma unroll
          for (int c = 0; c < 8; c++) {
            if (c0 + c < rem) g[(long)(c0 + c) * ld] = a[c];
          }
        }
      }
    }
    __syncthreads();
  }
}

// Apply the panel's row interchanges (rows j0..j0+nb-1) to columns [c_begin, c_end) of M.
__global__ void LaswpKernel(int j0, int nb, const int* __restrict__ ipiv, double* M, long ld,
                            int c_begin, int c_end) {
  const int c = c_begin + blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= c_end) return;
  double* col = M + (long)c * ld;
  for (int i = 0; i < nb; i++) {
    const int r = j0 + i, p = ipiv[r];
    if (p != r) {
      const double t = col[r];
      col[r] = col[p];
      col[p] = t;
    }
  }
}

// perm[i] = source row of row i after applying all interchanges. Single CTA; perm built in smem.
__global__ void BuildPermKernel(int n, const int* __restrict__ ipiv, int* perm) {
  extern __shared__ int sp[];
  for (int i = threadIdx.x; i < n; i += blockDim.x) sp[i] = i;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 0; i < n; i++) {
      const int p = ipiv[i];
      if (p != i) {
        const int t = sp[i];
        sp[i] = sp[p];
        sp[p] = t;
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) perm[i] = sp[i];
}

// dst[i, c] = src[perm[i], c]
__global__ void GatherRowsKernel(int n, int nrhs, const int* __restrict__ perm,
                                 const double* __restrict__ src, long lds, double* dst, long ldd) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int c = blockIdx.y;
  if (i < n && c < nrhs) dst[(long)c * ldd + i] = src[(long)c * lds + perm[i]];
}

// Diagonal-block triangular solve with many right-hand sides. T: nb x nb block at (ld).
// UPPER == false: unit lower (L of LU);  UPPER == true: non-unit upper (U of LU).
// X: nb x nrhs block (ldx), CTA handles kRhsCols columns; thread (r = tid % 32 col, q) layout.
template <bool UPPER>
__global__ void __launch_bounds__(256) TrsmDiagKernel(int nb, const double* __restrict__ T, long ld,
                                                      double* X, long ldx, int nrhs) {
  extern __shared__ double s[];
  const int PT = nb + 1;
  double* st = s;            // st[c*PT + r] = T[r][c]
  double* sx = s + nb * PT;  // sx[r*(kRhsCols+1) + c]   (row-major so a row step is conflict free)
  constexpr int PX = kRhsCols + 1;
  const int tid = threadIdx.x;
  const int c0 = blockIdx.x * kRhsCols;
  const int nc = min(kRhsCols, nrhs - c0);
  for (int e = tid; e < nb * nb; e += 256) {
    const int r = e % nb, c = e / nb;
    st[c * PT + r] = T[(long)c * ld + r];
  }
  for (int e = tid; e < nb * kRhsCols; e += 256) {
    const int r = e % nb, c = e / nb;
    sx[r * PX + c] = (c < nc) ? X[(long)(c0 + c) * ldx + r] : 0.0;
  }
  __syncthreads();
  const int c = tid % kRhsCols;  // my RHS column
  const int q = tid / kRhsCols;  // row phase 0..7
  if (!UPPER) {
    for (int j = 0; j < nb; j++) {
      const double xj = sx[j * PX + c];  // unit diagonal
      for (int r = j + 1 + q; r < nb; r += 8) sx[r * PX + c] -= st[j * PT + r] * xj;
      __syncthreads();
    }
  } else {
    for (int j = nb - 1; j >= 0; j--) {
      if (q == 0) sx[j * PX + c] /= st[j * PT + j];
      __syncthreads();
      const double xj = sx[j * PX + c];
      for (int r = q; r < j; r += 8) sx[r * PX + c] -= st[j * PT + r] * xj;
      __syncthreads();
    }
  }
  for (int e = tid; e < nb * kRhsCols; e += 256) {
    const int r = e % nb, cc = e / nb;
    if (cc < nc) X[(long)(c0 + cc) * ldx + r] = sx[r * PX + cc];
  }
}

constexpr int kLuPanelSmemBytes = 200 * 1024;  // dynamic shared memory of LuPanelSmemKernel

void ConfigureOnce() {
  static std::atomic<unsigned long long> configured{0};
  if (!FirstUseOnCurrentDevice(configured)) return;
  const int bytes = (int)(sizeof(double) * (kSolveNB * (kSolveNB + 1) + kSolveNB * (kRhsCols + 1)));
  cudaFuncSetAttribute(TrsmDiagKernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  cudaFuncSetAttribute(TrsmDiagKernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  cudaFuncSetAttribute(BuildPermKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  cudaFuncSetAttribute(LuPanelSmemKernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, kLuPanelSmemBytes);
  cudaFuncSetAttribute(LuPanelSmemKernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, kLuPanelSmemBytes);
}

size_t TrsmSmem(int nb) {
  return sizeof(double) * ((size_t)nb * (nb + 1) + (size_t)nb * (kRhsCols + 1));
}

__global__ void ResetInfoKernel2(int* info) { *info = 0; }

}  // namespace

namespace {
// Side stream of LuFactor's look-ahead, separate from the Cholesky's.
thread_local LookAhead t_lu_lookahead;

void LaunchPanel(cudaStream_t s, int n, int j0, int nb, double* A, long lda, int* ipiv, int* info) {
  // sub-panel width by what fits on chip: 8 columns up to 3200 rows, 4 up to 6400, else the global-memory kernel
  const size_t rows = (size_t)(n - j0);
  CountLaunch();
  if (rows * 8 * sizeof(double) <= (size_t)kLuPanelSmemBytes) {
    LuPanelSmemKernel<8><<<1, 1024, rows * 8 * sizeof(double), s>>>(n, j0, nb, A, lda, ipiv, info);
  } else if (rows * 4 * sizeof(double) <= (size_t)kLuPanelSmemBytes) {
    LuPanelSmemKernel<4><<<1, 1024, rows * 4 * sizeof(double), s>>>(n, j0, nb, A, lda, ipiv, info);
  } else {
    LuPanelKernel<<<1, 1024, 0, s>>>(n, j0, nb, A, lda, ipiv, info);
  }
}

// Panel (j0, nb) -> columns [c0, c1) right of it: row interchanges, U12 = L11^{-1} A12, A22 -= L21 U12.
int ApplyPanel(cudaStream_t s, int n, int j0, int nb, double* A, long lda, const int* ipiv, int c0, int c1) {
  const int cols = c1 - c0;
  if (cols <= 0) return 0;
  CountLaunch(); LaswpKernel<<<(cols + 127) / 128, 128, 0, s>>>(j0, nb, ipiv, A, lda, c0, c1);
  double* A12 = A + (long)c0 * lda + j0;
  CountLaunch(); TrsmDiagKernel<false><<<(cols + kRhsCols - 1) / kRhsCols, 256, TrsmSmem(nb), s>>>(
      nb, A + (long)j0 * lda + j0, lda, A12, lda, cols);
  const int below = n - j0 - nb;
  if (below <= 0) return 0;
  const double* L21 = A + (long)j0 * lda + j0 + nb;
  return Dgemm(s, false, false, below, cols, nb, -1.0, L21, lda, 0, A12, lda, 0, 1.0, A12 + nb, lda, 0, 1, false);
}
}  // namespace

// In-place LU with partial pivoting: P A = L U. Right-looking with a look-ahead of one panel: after panel J the
// columns of panel J + 1 are updated first and that panel is factored on a high-priority side stream (one CTA: 32
// dependent pivot columns) WHILE the main stream applies panel J to everything right of it. Every entry receives
// the same operations in the same order as in the sequential schedule: the factors are bit-identical.
int LuFactor(cudaStream_t s, int n, double* A, long lda, int* ipiv, int* info) {
  ConfigureOnce();
  CountLaunch(); ResetInfoKernel2<<<1, 1, 0, s>>>(info);
  LookAhead& la = t_lu_lookahead;
  const bool ahead = n > 4 * kLuNB && la.Prepare();
  LaunchPanel(s, n, 0, min(kLuNB, n), A, lda, ipiv, info);
  for (int j0 = 0; j0 < n; j0 += kLuNB) {
    const int nb = min(kLuNB, n - j0);
    // panel (j0, nb) is factored and visible to the main stream here
    if (j0 > 0) {
      CountLaunch(); LaswpKernel<<<(j0 + 127) / 128, 128, 0, s>>>(j0, nb, ipiv, A, lda, 0, j0);
    }
    const int n0 = j0 + nb;  // first column of the next panel
    if (n0 >= n) break;
    const int nb1 = min(kLuNB, n - n0);
    int rc = ApplyPanel(s, n, j0, nb, A, lda, ipiv, n0, n0 + nb1);
    if (rc != 0) return rc;
    if (ahead) {
      cudaEventRecord(la.updated, s);
      cudaStreamWaitEvent(la.side, la.updated, 0);
      LaunchPanel(la.side, n, n0, nb1, A, lda, ipiv, info);
      cudaEventRecord(la.factored, la.side);
    } else {
      LaunchPanel(s, n, n0, nb1, A, lda, ipiv, info);
    }
    rc = ApplyPanel(s, n, j0, nb, A, lda, ipiv, n0 + nb1, n);
    if (rc != 0) return rc;
    if (ahead) cudaStreamWaitEvent(s, la.factored, 0);
  }
  return LaunchStatus();
}

// Solve with the factors: X = U^{-1} L^{-1} P B. `B` is overwritten by X; `tmp` holds n*nrhs
// doubles (ld n); `perm` holds n ints.
int LuSolveFactored(cudaStream_t s, int n, const double* LU, long lda, const int* ipiv, int nrhs,
                    double* B, long ldb, double* tmp, int* perm) {
  ConfigureOnce();
  CountLaunch(); BuildPermKernel<<<1, 1024, sizeof(int) * n, s>>>(n, ipiv, perm);
  {
    dim3 grid((n + 255) / 256, nrhs);
    CountLaunch(); GatherRowsKernel<<<grid, 256, 0, s>>>(n, nrhs, perm, B, ldb, tmp, n);
  }
  // forward, unit lower
  for (int j0 = 0; j0 < n; j0 += kSolveNB) {
    const int nb = min(kSolveNB, n - j0);
    CountLaunch(); TrsmDiagKernel<false><<<(nrhs + kRhsCols - 1) / kRhsCols, 256, TrsmSmem(nb), s>>>(
        nb, LU + (long)j0 * lda + j0, lda, tmp + j0, n, nrhs);
    const int rest = n - j0 - nb;
    if (rest > 0) {
      const int rc = Dgemm(s, false, false, rest, nrhs, nb, -1.0, LU + (long)j0 * lda + j0 + nb, lda,
                           0, tmp + j0, n, 0, 1.0, tmp + j0 + nb, n, 0, 1, false);
      if (rc != 0) return rc;
    }
  }
  // backward, upper
  const int nblk = (n + kSolveNB - 1) / kSolveNB;
  for (int k = nblk - 1; k >= 0; k--) {
    const int j0 = k * kSolveNB, nb = min(kSolveNB, n - j0);
    CountLaunch(); TrsmDiagKernel<true><<<(nrhs + kRhsCols - 1) / kRhsCols, 256, TrsmSmem(nb), s>>>(
        nb, LU + (long)j0 * lda + j0, lda, tmp + j0, n, nrhs);
    if (j0 > 0) {
      const int rc = Dgemm(s, false, false, j0, nrhs, nb, -1.0, LU + (long)j0 * lda, lda, 0,
                           tmp + j0, n, 0, 1.0, tmp, n, 0, 1, false);
      if (rc != 0) return rc;
    }
  }
  // copy back
  cudaMemcpy2DAsync(B, sizeof(double) * ldb, tmp, sizeof(double) * n, sizeof(double) * n, nrhs,
                    cudaMemcpyDeviceToDevice, s);
  return LaunchStatus();
}

// out = pade33(X). work: 3*n*n doubles; iwork: 2*n ints.
int PadeExpm(cudaStream_t s, int n, const double* X, double* out, double* work, int* iwork,
             int* info) {
  const long nn = (long)n * n;
  double* P2 = work;           // X^2, then V
  double* T = work + nn;       // X^2 + 60 I, later LU scratch
  double* U = work + 2 * nn;   // odd part, then the denominator
  int rc = Dgemm(s, false, false, n, n, n, 1.0, X, n, 0, X, n, 0, 0.0, P2, n, 0, 1, false);
  if (rc) return rc;
  if ((rc = ScaleAddDiag(s, n, P2, 1.0, 60.0, T))) return rc;
  if ((rc = Dgemm(s, false, false, n, n, n, 1.0, X, n, 0, T, n, 0, 0.0, U, n, 0, 1, false))) return rc;
  if ((rc = ScaleAddDiag(s, n, P2, 12.0, 120.0, P2))) return rc;
  // out = V + U (numerator), U <- V - U (denominator)
  if ((rc = SumDiff(s, nn, U, P2, out, U))) return rc;
  if ((rc = LuFactor(s, n, U, n, iwork, info))) return rc;
  return LuSolveFactored(s, n, U, n, iwork, n, out, n, T, iwork + n);
}

}  // namespace cxb

using namespace cxb;

extern "C" {

size_t cxb_geodesic_worksize(int n) { return (size_t)4 * n * n; }

int cxb_lu_solve(void* stream, int n, double* dA, long lda, int nrhs, double* dB, long ldb,
                 int* d_ipiv, int* d_info) {
  // d_ipiv: 2n ints. Needs an n*nrhs scratch: allocate from the stream-ordered pool.
  cudaStream_t s = AsStream(stream);
  int rc = LuFactor(s, n, dA, lda, d_ipiv, d_info);
  if (rc) return rc;
  double* tmp = nullptr;
  if (cudaMallocAsync(&tmp, sizeof(double) * (size_t)n * nrhs, s) != cudaSuccess) return -1;
  rc = LuSolveFactored(s, n, dA, lda, d_ipiv, nrhs, dB, ldb, tmp, d_ipiv + n);
  cudaFreeAsync(tmp, s);
  return rc;
}

int cxb_pade_expm(void* stream, int n, const double* d_X, double* d_out, double* d_work,
                  int* d_iwork, int* d_info) {
  return PadeExpm(AsStream(stream), n, d_X, d_out, d_work, d_iwork, d_info);
}

int cxb_taylor_expm(void* stream, int n, const double* d_X, double* d_out, double* d_work) {
  // (I + X/4 + X^2/32)^4 — DoExponentialMap<1>, exponential_map.cc:15-42 (degree 2, 2 squarings)
  cudaStream_t s = AsStream(stream);
  double* Y = d_work;
  int rc = Dgemm(s, false, false, n, n, n, 1.0 / 32.0, d_X, n, 0, d_X, n, 0, 0.0, d_out, n, 0, 1, false);
  if (rc) return rc;
  if ((rc = ScaleAddDiag(s, n, d_X, 0.25, 1.0, Y))) return rc;                 // Y = I + X/4
  if ((rc = cxb_axpbypcz(stream, (long)n * n, 1.0, d_out, 1.0, Y, 0.0, nullptr))) return rc;  // + X^2/32
  if ((rc = Dgemm(s, false, false, n, n, n, 1.0, Y, n, 0, Y, n, 0, 0.0, d_out, n, 0, 1, false))) return rc;
  if ((rc = Dgemm(s, false, false, n, n, n, 1.0, d_out, n, 0, d_out, n, 0, 0.0, Y, n, 0, 1, false))) return rc;
  cudaMemcpyAsync(d_out, Y, sizeof(double) * (size_t)n * n, cudaMemcpyDeviceToDevice, s);
  return LaunchStatus();
}

int cxb_geodesic_update_taylor(void* stream, int n, double* d_W, double* d_WS, double e_weight,
                               double scale, double* d_work) {
  // hermitian_psd.cc:9-31: W <- sym( exp_taylor( scale (WS + e I) ) W ). d_work: 2 n^2 doubles.
  cudaStream_t s = AsStream(stream);
  const long nn = (long)n * n;
  int rc = ShiftScale(s, n, d_WS, e_weight, scale);
  if (rc) return rc;
  double* E = d_work + nn;
  if ((rc = cxb_taylor_expm(stream, n, d_WS, E, d_work))) return rc;
  if ((rc = Dgemm(s, false, false, n, n, n, 1.0, E, n, 0, d_W, n, 0, 0.0, d_WS, n, 0, 1, false))) return rc;
  cudaMemcpyAsync(d_W, d_WS, sizeof(double) * nn, cudaMemcpyDeviceToDevice, s);
  return Symmetrize(s, n, d_W);
}

int cxb_geodesic_update(void* stream, int n, double* d_W, double* d_WS, double e_weight,
                        double scale, double* d_work, int* d_iwork, int* d_info) {
  cudaStream_t s = AsStream(stream);
  const long nn = (long)n * n;
  int rc = ShiftScale(s, n, d_WS, e_weight, scale);
  if (rc) return rc;
  double* E = d_work + 3 * nn;
  if ((rc = PadeExpm(s, n, d_WS, E, d_work, d_iwork, d_info))) return rc;
  // W <- E W (into d_WS as scratch), then symmetrise.
  if ((rc = Dgemm(s, false, false, n, n, n, 1.0, E, n, 0, d_W, n, 0, 0.0, d_WS, n, 0, 1, false)))
    return rc;
  cudaMemcpyAsync(d_W, d_WS, sizeof(double) * nn, cudaMemcpyDeviceToDevice, s);
  return Symmetrize(s, n, d_W);
}

}  // extern "C"

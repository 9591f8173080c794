// K3 / K5: blocked right-looking Cholesky of the dense Schur complement and the triangular solves.
//
// Replaces BlockCholeskyInPlace / ApplyBlockInverse(OfTranspose)InPlace
// (block_triangular_operations.cc:114-219) for one dense supernode.
//
// Factorisation, two levels of blocking:
//   outer block column of kOuter = 512 columns:
//     for each inner block of kNB = 128 columns inside it
//       1. PotrfDiagBlockedKernel — one CTA factors the 128 x 128 diagonal block in shared memory,
//                             in 32 x 32 sub-blocks (warp-shuffle factor of the diagonal part,
//                             substitution for the rows below, register-tiled rank-32 update);
//       2. TrsmPanelKernel  — X L11^T = A21 by true substitution (no explicit inverses: H becomes
//                             very ill conditioned late in the IPM). One thread per row keeps 32
//                             accumulators in registers; L11 is streamed through shared memory in
//                             32-column slabs and read as 16-byte broadcasts;
//       3. DMMA update of the rest of the outer block column (lower trapezoid, K = 128);
//     DMMA SYRK of everything to the right with K = 512 (gemm.cu) — where the flops are.
// Above 3 x 512 columns the outer loop runs with a look-ahead of one block column: panel J + 1 is
// factored on a high-priority side stream while panel J updates the rest of the trailing matrix.
// A non-positive pivot sets *info = 1 + column (Eigen::LLT::info() != Success in the reference).
//
// Solves: one launch per sweep and right-hand side, a wavefront over the 128-row blocks whose
// hand-off between CTAs is the solution vector itself, polled against a sentinel (see "triangular
// solves" below).
//
// The LDL^T (K4) reuses the panel solve and the DMMA updates; its diagonal blocks are factored by
// LdltDiagKernel, a signed rank-1 variant (L S L^T, S = diag(+-1)).
// All global->shared staging keeps 8 loads in flight per thread (latency, not bandwidth, is the
// limit of these small kernels).
#include <algorithm>
#include "common.cuh"
#include "device_api.h"

namespace cxb {
namespace {

constexpr int kNB = 128;     // inner block
constexpr int kOuter = 512;  // outer block column (K of the big SYRK)
constexpr int kMaxRhs = 4;

// Global -> shared staging with U loads in flight per thread (a plain load/store loop exposes the
// full memory latency once per element).
template <int U, typename LoadF, typename StoreF>
__device__ __forceinline__ void BatchedCopy(int total, int tid, int nthreads, LoadF load, StoreF store) {
  for (int base = tid; base < total; base += nthreads * U) {
    double v[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const int e = base + u * nthreads;
      v[u] = (e < total) ? load(e) : 0.0;
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const int e = base + u * nthreads;
      if (e < total) store(e, v[u]);
    }
  }
}

// ---- 1. diagonal block ---------------------------------------------------------------------------
// Signed factorisation of the nb x nb (nb <= 128) block at H (ld) in place, lower triangle: a symmetric
// indefinite block becomes L S L^T with S = diag(+-1) ("signed Cholesky" = LDL^T with D = S and the
// columns of L scaled by sqrt|d|), S stored to signs[col0 ..]. Pivots with |d| <= 1e-9 are replaced by
// +-1e-9 like Eigen::RLDLT (RLDLT.h:378-389) and reported through info[1]; it never fails.
// One CTA of 512 threads, column scale + rank-1 update per step: thread t owns row r = t % 128 and the
// columns c with c % 4 == t / 128.
__global__ void __launch_bounds__(512) LdltDiagKernel(int nb, double* H, long ld, int col0, int* info,
                                                      double* signs) {
  extern __shared__ double s[];  // s[c * P + r], P = 129
  constexpr int P = kNB + 1;
  const int tid = threadIdx.x;
  const int r = tid & (kNB - 1);
  const int cg = tid >> 7;  // 0..3
  BatchedCopy<8>(
      kNB * kNB, tid, 512,
      [&](int e) {
        const int rr = e & (kNB - 1), c = e >> 7;
        return (rr < nb && c <= rr) ? H[(long)c * ld + rr] : 0.0;
      },
      [&](int e, double v) { s[(e >> 7) * P + (e & (kNB - 1))] = v; });
  __syncthreads();
  for (int j = 0; j < nb; j++) {
    double d = s[j * P + j];
    if (!(fabs(d) > 1e-9)) {
      d = (d < 0) ? -1e-9 : 1e-9;
      if (tid == 0) info[1] = 1;  // regularization_used
    }
    const double sign = (d < 0) ? -1.0 : 1.0;
    if (tid == 0) signs[col0 + j] = sign;
    d = fabs(d);
    const double rd = sqrt(d);
    const double inv = 1.0 / rd;
    // l[r] for this thread's row (pre-scale value is still in s[j][r] until the barrier below);
    // column j of L is sign * a_j / sqrt|d| and the update is sign * (a_r a_c / |d|)
    const double lr = (r > j && r < nb) ? s[j * P + r] * inv : 0.0;
    // trailing update of my row: s[c][r] -= l[r] * l[c] for j < c <= r, c in my column group
    if (r > j && r < nb) {
      int c = j + 1 + ((cg - (j + 1)) & 3);  // first c > j with c % 4 == cg
      const double slr = sign * lr;
      for (; c <= r; c += 4) s[c * P + r] -= slr * (s[j * P + c] * inv);
    }
    __syncthreads();  // all reads of the unscaled column j are done
    if (cg == 0 && r < nb) {
      if (r == j) s[j * P + j] = rd;
      if (r > j) s[j * P + r] = sign * lr;
    }
    __syncthreads();
  }
  __syncthreads();
  if (r < nb) {
    for (int c = cg; c <= r; c += 4) H[(long)c * ld + r] = s[c * P + r];
  }
}

// Cholesky of the diagonal block, blocked 32 x 32 inside the CTA (a rank-1 kernel like the one above
// spends two barriers per column: 132 us per 128 x 128 block, 40 % of the whole factorisation at m = 10^4):
//   for each 32-column sub-block: warp 0 factors the 32 x 32 diagonal part in registers (lane = row,
//   column entries exchanged by shuffles); one thread per row below solves its 32 entries by
//   substitution in registers; all 512 threads apply the rank-32 update to the rest of the block
//   with 3 x 6 register tiles (rows by lane: conflict-free, columns by warp: broadcast).
__global__ void __launch_bounds__(512) PotrfDiagBlockedKernel(int nb, double* H, long ld, int col0, int* info) {
  extern __shared__ double s[];  // s[c * P + r], P = 129
  constexpr int P = kNB + 1;
  constexpr unsigned kFull = 0xffffffffu;
  __shared__ int failed;
  __shared__ double srd[32];  // reciprocal diagonal of the current sub-block
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (*info != 0) return;  // an earlier block already failed
  if (tid == 0) failed = 0;
  BatchedCopy<8>(
      kNB * kNB, tid, 512,
      [&](int e) {
        const int rr = e & (kNB - 1), c = e >> 7;
        if (rr >= nb) return (c == rr) ? 1.0 : 0.0;  // identity padding keeps the arithmetic harmless
        return (c <= rr) ? H[(long)c * ld + rr] : 0.0;
      },
      [&](int e, double v) { s[(e >> 7) * P + (e & (kNB - 1))] = v; });
  __syncthreads();
  for (int k0 = 0; k0 < nb; k0 += 32) {
    // 1. diagonal sub-block
    if (warp == 0) {
      double a[32];
#pragma unroll
      for (int c = 0; c < 32; c++) a[c] = s[(k0 + c) * P + k0 + lane];
      int bad = 0;
#pragma unroll
      for (int j = 0; j < 32; j++) {
        const double d = __shfl_sync(kFull, a[j], j);
        if (!(d > 0.0) && bad == 0) bad = j + 1;  // same d in every lane
        const double rd = sqrt(d);
        const double inv = 1.0 / rd;
        const double l = (lane > j) ? a[j] * inv : ((lane == j) ? rd : 0.0);
        a[j] = l;
        if (lane == j) srd[j] = inv;
#pragma unroll
        for (int c = j + 1; c < 32; c++) {
          const double lc = __shfl_sync(kFull, l, c);
          a[c] -= l * lc;  // entries above the diagonal (c > lane) are never read again
        }
      }
#pragma unroll
      for (int c = 0; c < 32; c++) {
        if (c <= lane) s[(k0 + c) * P + k0 + lane] = a[c];
      }
      if (bad != 0 && lane == 0) {
        failed = 1;
        *info = col0 + k0 + bad;
      }
    }
    __syncthreads();
    if (failed) return;
    const int base = k0 + 32;
    const int below = kNB - base;  // rows base .. 127 (padded rows are zero)
    if (below == 0) break;
    // 2. rows below: x D^T = a, one thread per row
    if (tid < below) {
      const int r = base + tid;
      double x[32];
#pragma unroll
      for (int c = 0; c < 32; c++) x[c] = s[(k0 + c) * P + r];
#pragma unroll
      for (int c = 0; c < 32; c++) {
        const double xc = x[c] * srd[c];
        x[c] = xc;
        const double* dcol = s + (k0 + c) * P + k0;  // D[cq][c], cq > c
#pragma unroll
        for (int cq = c + 1; cq < 32; cq++) x[cq] -= xc * dcol[cq];
      }
#pragma unroll
      for (int c = 0; c < 32; c++) s[(k0 + c) * P + r] = x[c];
    }
    __syncthreads();
    // 3. rank-32 update of the trailing part: rows base + lane + 32 a, columns base + warp + 16 b
    {
      const int na = below >> 5, nbcol = below >> 4;  // 3 / 6, 2 / 4, 1 / 2
      double acc[3][6];
#pragma unroll
      for (int a = 0; a < 3; a++) {
#pragma unroll
        for (int b = 0; b < 6; b++) acc[a][b] = 0.0;
      }
      for (int k = 0; k < 32; k++) {
        const double* xk = s + (k0 + k) * P + base;
        double xr[3], xc[6];
#pragma unroll
        for (int a = 0; a < 3; a++) xr[a] = (a < na) ? xk[lane + 32 * a] : 0.0;
#pragma unroll
        for (int b = 0; b < 6; b++) xc[b] = (b < nbcol) ? xk[warp + 16 * b] : 0.0;
#pragma unroll
        for (int a = 0; a < 3; a++) {
#pragma unroll
          for (int b = 0; b < 6; b++) acc[a][b] += xr[a] * xc[b];
        }
      }
#pragma unroll
      for (int a = 0; a < 3; a++) {
#pragma unroll
        for (int b = 0; b < 6; b++) {
          const int r = base + lane + 32 * a, c = base + warp + 16 * b;
          if (a < na && b < nbcol && c <= r) s[c * P + r] -= acc[a][b];
        }
      }
    }
    __syncthreads();
  }
  const int r = tid & (kNB - 1), cg = tid >> 7;
  if (r < nb) {
    for (int c = cg; c <= r; c += 4) H[(long)c * ld + r] = s[c * P + r];
  }
}

// ---- 2. panel solve ---------------------------------------------------------------------------------
// Solves X * L11^T = A21 for kNB-row strips: one thread per row. L11: nb x nb lower (ld), nb <= 128.
// A21 (ld) is overwritten by X. Shared memory: sx[i][row] (the row's solved entries) and one slab of
// L11 rows, sl[i][c'] = L11[c0 + c'][i] for the 32 columns c0.. of the current phase.
__global__ void __launch_bounds__(kNB) TrsmPanelKernel(int nb, const double* __restrict__ L11, long ld,
                                                      double* A21, int rows, const int* info) {
  extern __shared__ __align__(16) double sm[];
  if (*info != 0) return;
  double* sx = sm;                 // [kNB][kNB]: sx[i * kNB + t]
  double* sl = sm + kNB * kNB;     // [kNB][32]:  sl[i * 32 + c']
  double* srd = sl + kNB * 32;     // [32] reciprocal diagonal of the current slab
  const int t = threadIdx.x;
  const int row = blockIdx.x * kNB + t;
  const bool active = row < rows;
  for (int c0 = 0; c0 < nb; c0 += 32) {
    const int cw = min(32, nb - c0);
    __syncthreads();
    // slab: columns i < c0 + cw of rows c0 .. c0 + cw - 1 of L11 (zero beyond the diagonal)
    BatchedCopy<8>(
        (c0 + 32) * 32, t, kNB,
        [&](int e) {
          const int cp = e & 31, i = e >> 5;
          const int c = c0 + cp;
          return (cp < cw && i <= c) ? L11[(long)i * ld + c] : 0.0;
        },
        [&](int e, double v) { sl[e] = v; });
    if (t < 32) srd[t] = (t < cw) ? 1.0 / L11[(long)(c0 + t) * ld + c0 + t] : 0.0;
    double acc[32];
#pragma unroll
    for (int cp = 0; cp < 32; cp++) {
      acc[cp] = (active && cp < cw) ? A21[(long)(c0 + cp) * ld + row] : 0.0;
    }
    __syncthreads();
    // acc[c'] -= sum_{i < c0} x_i L11[c0 + c'][i]
    for (int i = 0; i < c0; i++) {
      const double xi = sx[i * kNB + t];
      const double2* lrow = reinterpret_cast<const double2*>(sl + i * 32);
#pragma unroll
      for (int q = 0; q < 16; q++) {
        const double2 l = lrow[q];
        acc[2 * q] -= xi * l.x;
        acc[2 * q + 1] -= xi * l.y;
      }
    }
    // 32 x 32 diagonal block by substitution in registers
#pragma unroll
    for (int cp = 0; cp < 32; cp++) {
      const double x = acc[cp] * srd[cp];
      acc[cp] = x;
      const double* lrow = sl + (c0 + cp) * 32;  // L11[c0 + c''][c0 + cp] for c'' > cp
#pragma unroll
      for (int cq = cp + 1; cq < 32; cq++) acc[cq] -= x * lrow[cq];
    }
#pragma unroll
    for (int cp = 0; cp < 32; cp++) {
      sx[(c0 + cp) * kNB + t] = acc[cp];
      if (active && cp < cw) A21[(long)(c0 + cp) * ld + row] = acc[cp];
    }
  }
}

// ---- triangular solves -------------------------------------------------------------------------------
// One launch per sweep and right-hand side: a wavefront over the 128-row blocks. The CTA with ticket i owns
// block row i of the sweep: it streams its own part of L exactly once, consuming each earlier solution block
// as soon as its owner has stored it, then solves its 128 x 128 diagonal block and stores x_i. Tickets come
// from an atomic counter, so a CTA only ever waits for CTAs that started before it: no co-residency
// assumption, no deadlock when m / 128 exceeds the number of SMs.
// The solution itself is the hand-off: the output vector is pre-filled with a sentinel (a quiet NaN with a
// payload no computation produces) and every consuming WARP polls the 32 (forward) / 128 (backward) solution
// entries it needs with relaxed gpu-scope loads until none is the sentinel: one L2 round trip, no flag, no
// fence (each entry is a single 64-bit store, so seeing it is seeing all of it) and no CTA barrier between
// the producer's store and the consumer's FMAs. (A release/acquire flag per block costs about 5 us of
// barriers, fence and spin per hand-off, and that chain of m / 128 hand-offs, not bandwidth, set the pace:
// profiles/r01_m_*.) The right-hand side is read from a separate array. The diagonal blocks are solved by
// true substitution, with the reciprocal of the diagonal folded into the rows beforehand so that the
// 32-step chain is shuffle + FMA only. Summation order is fixed: results are deterministic.
// Loads the nb x nb lower block L (ld) into shared memory, sl[c * P + r] = L[r][c], and the
// reciprocals of its diagonal into srd.
template <int P>
__device__ __forceinline__ void LoadLowerBlock(double* sl, double* srd, const double* __restrict__ L,
                                               long ld, int nb) {
  BatchedCopy<8>(
      kNB * kNB, threadIdx.x, blockDim.x,
      [&](int e) {
        const int r = e & (kNB - 1), c = e >> 7;
        return (r < nb && c <= r) ? L[(long)c * ld + r] : 0.0;
      },
      [&](int e, double v) { sl[(e >> 7) * P + (e & (kNB - 1))] = v; });
  if (threadIdx.x < kNB) {
    srd[threadIdx.x] = (threadIdx.x < nb) ? 1.0 / L[(long)threadIdx.x * ld + threadIdx.x] : 0.0;
  }
}

constexpr unsigned long long kSentinelBits = 0x7FF8DEADBEEF0001ull;
__device__ __forceinline__ bool IsSentinel(double v) {
  return static_cast<unsigned long long>(__double_as_longlong(v)) == kSentinelBits;
}
__device__ __forceinline__ double LoadRelaxed(const double* p) {
  double v;
  asm volatile("ld.relaxed.gpu.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void StoreRelaxed(double* p, double v) {
  asm volatile("st.relaxed.gpu.global.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}

__global__ void WaveInitKernel(double* out, long count, int* tickets, int ntickets) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) out[i] = __longlong_as_double(static_cast<long long>(kSentinelBits));
  if (i < ntickets) tickets[i] = 0;
}

template <int P>
__device__ __forceinline__ void SolveLowerBlockScaled(const double* sl, const double* srd, double* sx) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#pragma unroll 1
  for (int b0 = 0; b0 < kNB; b0 += 32) {
    if (warp == 0) {
      const double rd = srd[b0 + lane];
      double lrow[32];
#pragma unroll
      for (int j = 0; j < 32; j++) lrow[j] = sl[(b0 + j) * P + b0 + lane] * rd;  // L[b0 + lane][b0 + j] / L_rr
      double v = sx[b0 + lane] * rd;
#pragma unroll
      for (int j = 0; j < 32; j++) {
        const double xj = __shfl_sync(0xffffffffu, v, j);
        if (lane > j) v -= lrow[j] * xj;
      }
      sx[b0 + lane] = v;
    }
    __syncthreads();
    const int rows = kNB - b0 - 32;
    if (tid < rows * 4) {
      const int r = b0 + 32 + (tid >> 2), q = tid & 3;
      double a = 0;
#pragma unroll
      for (int j = 0; j < 8; j++) a += sl[(b0 + q * 8 + j) * P + r] * sx[b0 + q * 8 + j];
      a += __shfl_xor_sync(0xffffffffu, a, 1);
      a += __shfl_xor_sync(0xffffffffu, a, 2);
      if (q == 0) sx[r] -= a;
    }
    __syncthreads();
  }
}

template <int P>
__device__ __forceinline__ void SolveLowerTransposedBlockScaled(const double* sl, const double* srd, double* sx) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#pragma unroll 1
  for (int b0 = kNB - 32; b0 >= 0; b0 -= 32) {
    if (warp == 0) {
      const double rd = srd[b0 + lane];
      double lcol[32];
#pragma unroll
      for (int j = 0; j < 32; j++) lcol[j] = sl[(b0 + lane) * P + b0 + j] * rd;  // L[b0 + j][b0 + lane] / L_cc
      double v = sx[b0 + lane] * rd;
#pragma unroll
      for (int j = 31; j >= 0; j--) {
        const double xj = __shfl_sync(0xffffffffu, v, j);
        if (lane < j) v -= lcol[j] * xj;
      }
      sx[b0 + lane] = v;
    }
    __syncthreads();
    if (tid < b0 * 4) {
      const int r = tid >> 2, q = tid & 3;
      double a = 0;
#pragma unroll
      for (int j = 0; j < 8; j++) a += sl[r * P + b0 + q * 8 + j] * sx[b0 + q * 8 + j];
      a += __shfl_xor_sync(0xffffffffu, a, 1);
      a += __shfl_xor_sync(0xffffffffu, a, 2);
      if (q == 0) sx[r] -= a;
    }
    __syncthreads();
  }
}

// Out must be sentinel-filled and *ticket zero at launch; B (the right-hand side) is not written.
__global__ void __launch_bounds__(512) TrsvFwdPollKernel(int m, const double* __restrict__ L, long ld,
                                                         const double* __restrict__ B, double* Out, int* ticket) {
  constexpr int P = kNB + 1;
  extern __shared__ double s[];
  double* sl = s;
  double* sx = s + kNB * P;
  double* srd = sx + kNB;
  double* sp = srd + kNB;  // 4 x kNB partial sums
  __shared__ int s_block;
  const int tid = threadIdx.x, lane = tid & 31;
  if (tid == 0) s_block = atomicAdd(ticket, 1);
  __syncthreads();
  const int i = s_block;
  const int r0 = i * kNB;
  const int nb = min(kNB, m - r0);
  LoadLowerBlock<P>(sl, srd, L + (long)r0 * ld + r0, ld, nb);
  const int rl = tid & (kNB - 1), g = tid >> 7;  // row of the strip, column group (32 of every 128)
  const bool active = rl < nb;
  const int r = r0 + rl;
  double acc = 0;
  for (int kb = 0; kb < i; kb++) {
    const double* Lr = L + (long)(kb * kNB + g * 32) * ld + r;
    double l[32];
#pragma unroll
    for (int c = 0; c < 32; c++) l[c] = active ? __ldcs(Lr + (long)c * ld) : 0.0;  // read exactly once
    const double* xp = Out + kb * kNB + g * 32 + lane;  // blocks kb < i are full: always < m
    double xv;
    do {
      xv = LoadRelaxed(xp);
    } while (__any_sync(0xffffffffu, IsSentinel(xv)));
#pragma unroll
    for (int c = 0; c < 32; c++) acc += l[c] * __shfl_sync(0xffffffffu, xv, c);
  }
  sp[g * kNB + rl] = acc;
  __syncthreads();
  if (g == 0) sx[rl] = active ? B[r] - (((sp[rl] + sp[kNB + rl]) + sp[2 * kNB + rl]) + sp[3 * kNB + rl]) : 0.0;
  __syncthreads();
  SolveLowerBlockScaled<P>(sl, srd, sx);
  if (tid < nb) StoreRelaxed(Out + r0 + tid, sx[tid]);
}

__global__ void __launch_bounds__(512) TrsvBwdPollKernel(int m, const double* __restrict__ L, long ld,
                                                         const double* __restrict__ B, double* Out, int* ticket) {
  constexpr int P = kNB + 1;
  extern __shared__ double s[];
  double* sl = s;
  double* sx = s + kNB * P;
  double* srd = sx + kNB;
  double* sp = srd + kNB;  // kNB column sums
  __shared__ int s_block;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_block = atomicAdd(ticket, 1);
  __syncthreads();
  const int nblk = (m + kNB - 1) / kNB;
  const int i = nblk - 1 - s_block;
  const int c0 = i * kNB;
  const int nb = min(kNB, m - c0);
  LoadLowerBlock<P>(sl, srd, L + (long)c0 * ld + c0, ld, nb);
  // warp w owns the columns c0 + 8 w .. c0 + 8 w + 7 of L; lanes run down the rows of a block
  double acc[8];
#pragma unroll
  for (int q = 0; q < 8; q++) acc[q] = 0;
  for (int kb = nblk - 1; kb > i; kb--) {
    const int rb = kb * kNB;
    const int nrows = min(kNB, m - rb);
    double l[8][4];
#pragma unroll
    for (int q = 0; q < 8; q++) {
      const int cw = warp * 8 + q;
      const double* Lc = L + (long)(c0 + cw) * ld + rb + lane;
#pragma unroll
      for (int p = 0; p < 4; p++) l[q][p] = (cw < nb && lane + 32 * p < nrows) ? __ldcs(Lc + 32 * p) : 0.0;
    }
    double xv[4];
    bool pending;
    do {
      pending = false;
#pragma unroll
      for (int p = 0; p < 4; p++) {
        if (lane + 32 * p < nrows) {
          xv[p] = LoadRelaxed(Out + rb + lane + 32 * p);
          pending = pending || IsSentinel(xv[p]);
        } else {
          xv[p] = 0.0;
        }
      }
    } while (__any_sync(0xffffffffu, pending));
#pragma unroll
    for (int q = 0; q < 8; q++) {
#pragma unroll
      for (int p = 0; p < 4; p++) acc[q] += l[q][p] * xv[p];
    }
  }
#pragma unroll
  for (int q = 0; q < 8; q++) {
    const double v = WarpSum(acc[q]);
    if (lane == 0) sp[warp * 8 + q] = v;
  }
  __syncthreads();
  if (tid < kNB) sx[tid] = (tid < nb) ? B[c0 + tid] - sp[tid] : 0.0;
  __syncthreads();
  SolveLowerTransposedBlockScaled<P>(sl, srd, sx);
  if (tid < nb) StoreRelaxed(Out + c0 + tid, sx[tid]);
}

// ---- supernodal (multifrontal) pieces -----------------------------------------------------------------
// dst[idx[e]] += sign * G[a, b] for the pairs a >= b of an n x n lower triangle, e = position of (a, b)
// in column-major order of the lower triangle. idx < 0: entry dropped.
__global__ void ScatterLowerIndexedKernel(int n, const double* __restrict__ G, long ldg,
                                          const long* __restrict__ idx, double sign, double* dst) {
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (a >= n || a < b) return;
  const long e = (long)b * n - (long)b * (b - 1) / 2 + (a - b);
  const long d = idx[e];
  if (d >= 0) dst[d] += sign * G[(long)b * ldg + a];
}

// Forward pass of one front: x[sep[r]] -= sum_c L21[r][c] xk[c], one warp per separator row.
__global__ void FrontForwardKernel(int p, int sk, const double* __restrict__ L21, long ld,
                                   const double* __restrict__ xk, const int* __restrict__ sep, double* x) {
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= p) return;
  double a = 0;
  for (int c = lane; c < sk; c += 32) a += L21[(long)c * ld + r] * xk[c];
  a = WarpSum(a);
  if (lane == 0) x[sep[r]] -= a;
}

// Backward pass of one front: xk[c] -= sum_r L21[r][c] x[sep[r]], one warp per column.
__global__ void FrontBackwardKernel(int p, int sk, const double* __restrict__ L21, long ld, double* xk,
                                    const int* __restrict__ sep, const double* __restrict__ x) {
  const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (c >= sk) return;
  double a = 0;
  for (int r = lane; r < p; r += 32) a += L21[(long)c * ld + r] * x[sep[r]];
  a = WarpSum(a);
  if (lane == 0) xk[c] -= a;
}

__global__ void ResetInfoKernel(int* info) { *info = 0; }
__global__ void ResetInfo2Kernel(int* info) { info[0] = 0; info[1] = 0; }

// After the panel solve Y = A21 L11^{-T} of the signed factorisation: keeps Y in `Yout` (rows x nb,
// ld = rows) for the trailing update A22 -= Y (Y S)^T and stores L21 = Y S in place.
__global__ void SignedPanelKernel(int rows, int nb, double* A21, long ld, const double* __restrict__ signs,
                                  double* Yout) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  const int c = blockIdx.y;
  if (r >= rows || c >= nb) return;
  const double y = A21[(long)c * ld + r];
  Yout[(long)c * rows + r] = y;
  A21[(long)c * ld + r] = y * signs[c];
}

// Kp[i][j] = K[max(pi, pj)][min(pi, pj)], i >= j: the symmetric permutation P K P^T of a matrix
// stored by its lower triangle.
__global__ void SymPermuteLowerKernel(int N, const double* __restrict__ K, long ldk,
                                      const int* __restrict__ perm, double* Kp, long ldp) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int j = blockIdx.y;
  if (i >= N || i < j) return;
  const int pi = perm[i], pj = perm[j];
  const int r = pi > pj ? pi : pj, c = pi > pj ? pj : pi;
  Kp[(long)j * ldp + i] = K[(long)c * ldk + r];
}

// A front (rows x s lower trapezoid: the s x s diagonal block stored by its lower triangle on top of the
// (rows - s) x s separator block) under the pivot order `perm` of its supernode: the diagonal block becomes
// P F11 P^T, the separator block gets its columns permuted.
__global__ void FrontPermuteKernel(int rows, int s, const double* __restrict__ F, long ld,
                                   const int* __restrict__ perm, double* Out, long ldo) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  const int c = blockIdx.y;
  if (r >= rows || r < c) return;
  const int pc = perm[c];
  if (r < s) {
    const int pr = perm[r];
    const int a = pr > pc ? pr : pc, b = pr > pc ? pc : pr;
    Out[(long)c * ldo + r] = F[(long)b * ld + a];
  } else {
    Out[(long)c * ldo + r] = F[(long)pc * ld + r];
  }
}

// Out[:, c] = A[:, c] * signs[c]
__global__ void ScaleColumnsKernel(int rows, int cols, const double* __restrict__ A, long lda,
                                   const double* __restrict__ signs, double* Out, long ldo) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  const int c = blockIdx.y;
  if (r >= rows || c >= cols) return;
  Out[(long)c * ldo + r] = A[(long)c * lda + r] * signs[c];
}

// out[i] = in[perm[i]] (gather) or out[perm[i]] = in[i] (scatter)
__global__ void PermuteVecKernel(int N, const int* __restrict__ perm, const double* __restrict__ in,
                                 double* out, int scatter) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  if (scatter) {
    out[perm[i]] = in[i];
  } else {
    out[i] = in[perm[i]];
  }
}

__global__ void ApplySignsKernel(int N, int nrhs, const double* __restrict__ signs, double* Z, long ldz) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  for (int k = 0; k < nrhs; k++) Z[(long)k * ldz + i] *= signs[i];
}

constexpr size_t kDiagSmem = sizeof(double) * kNB * (kNB + 1);
constexpr size_t kTrsmSmem = sizeof(double) * (kNB * kNB + kNB * 32 + 32);
constexpr size_t kWaveSmem = sizeof(double) * (kNB * (kNB + 1) + 8 * kNB);

void ConfigureOnce() {
  static std::atomic<unsigned long long> configured{0};
  if (!FirstUseOnCurrentDevice(configured)) return;
  cudaFuncSetAttribute(LdltDiagKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDiagSmem);
  cudaFuncSetAttribute(PotrfDiagBlockedKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDiagSmem);
  cudaFuncSetAttribute(TrsmPanelKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTrsmSmem);
  cudaFuncSetAttribute(TrsvFwdPollKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWaveSmem);
  cudaFuncSetAttribute(TrsvBwdPollKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWaveSmem);
}

}  // namespace

// Factors the block column [j0, j0 + w) x rows [j0, m) of H in place (w <= kOuter): inner
// right-looking steps of kNB columns whose updates stay inside the block column.
int PotrfBlockColumn(cudaStream_t s, int m, int j0, int w, double* H, long ldh, int* info) {
  ConfigureOnce();
  for (int i0 = j0; i0 < j0 + w; i0 += kNB) {
    const int nb = min(kNB, j0 + w - i0);
    double* Hii = H + (long)i0 * ldh + i0;
    CountLaunch(); PotrfDiagBlockedKernel<<<1, 512, kDiagSmem, s>>>(nb, Hii, ldh, i0, info);
    const int rows = m - i0 - nb;
    if (rows <= 0) continue;
    double* A21 = Hii + nb;
    CountLaunch(); TrsmPanelKernel<<<(rows + kNB - 1) / kNB, kNB, kTrsmSmem, s>>>(nb, Hii, ldh, A21, rows, info);
    const int rest = j0 + w - (i0 + nb);  // columns of this block column still to be updated
    if (rest > 0) {
      // trapezoid: rows i0+nb .. m-1, columns i0+nb .. j0+w-1 (lower part)
      const int rc = DgemmEx(s, -1, 1, false, true, rows, rest, nb, -1.0, A21, ldh, 0, A21, ldh, 0, 1.0,
                             H + (long)(i0 + nb) * ldh + (i0 + nb), ldh, 0, 1, true, false, 0);
      if (rc != 0) return rc;
    }
  }
  return LaunchStatus();
}

}  // namespace cxb

using namespace cxb;

extern "C" {

size_t cxb_potrf_worksize(int m) {
  (void)m;
  return 1;  // the algorithm works fully in place
}

namespace {
// Side stream of the Cholesky's look-ahead below, separate from the LU's.
thread_local LookAhead t_lookahead;

// Right-looking factorisation with a look-ahead of one outer block column: after panel J the update
// of block column J + 1 is issued first, panel J + 1 is then factored on a high-priority side stream
// (its chain of small latency-bound kernels: 4 x {diagonal block, panel solve, in-panel update})
// WHILE the main stream applies panel J to the rest of the trailing matrix on the tensor cores.
// Every entry still receives the same updates in the same order: the factor is bit-identical to the
// sequential schedule's.
int PotrfLookAhead(cudaStream_t s, int m, double* dH, long ldh, int* d_info) {
  LookAhead& la = t_lookahead;
  if (!la.Prepare()) return (int)cudaErrorUnknown;
  int rc = PotrfBlockColumn(s, m, 0, min(kOuter, m), dH, ldh, d_info);
  if (rc != 0) return rc;
  for (int j0 = 0; j0 < m; j0 += kOuter) {
    const int w = min(kOuter, m - j0);
    const int rows = m - j0 - w;
    if (rows <= 0) break;
    const int n0 = j0 + w;               // first column of the next panel
    const int wn = min(kOuter, rows);    // its width
    const double* L21 = dH + (long)j0 * ldh + n0;
    double* A22 = dH + (long)n0 * ldh + n0;
    // 1. panel J -> block column J + 1 (lower trapezoid, rows x wn)
    rc = Dgemm(s, false, true, rows, wn, w, -1.0, L21, ldh, 0, L21, ldh, 0, 1.0, A22, ldh, 0, 1, true);
    if (rc != 0) return rc;
    cudaEventRecord(la.updated, s);
    cudaStreamWaitEvent(la.side, la.updated, 0);
    // 2. factor panel J + 1 on the side stream
    rc = PotrfBlockColumn(la.side, m, n0, wn, dH, ldh, d_info);
    if (rc != 0) return rc;
    cudaEventRecord(la.factored, la.side);
    // 3. panel J -> everything right of block column J + 1
    const int rest = rows - wn;
    if (rest > 0) {
      rc = Dgemm(s, false, true, rest, rest, w, -1.0, L21 + wn, ldh, 0, L21 + wn, ldh, 0, 1.0,
                 A22 + (long)wn * ldh + wn, ldh, 0, 1, true);
      if (rc != 0) return rc;
    }
    cudaStreamWaitEvent(s, la.factored, 0);
  }
  return LaunchStatus();
}
}  // namespace

int cxb_potrf_lower(void* stream, int m, double* dH, long ldh, double* d_work, int* d_info) {
  (void)d_work;
  cudaStream_t s = AsStream(stream);
  if (m <= 0) return 0;
  CountLaunch(); ResetInfoKernel<<<1, 1, 0, s>>>(d_info);
  // below three outer block columns there is nothing to overlap; the legacy default stream cannot
  // run concurrently with a side stream's work ordering-wise in a useful way either
  if (m > 3 * kOuter) return PotrfLookAhead(s, m, dH, ldh, d_info);
  for (int j0 = 0; j0 < m; j0 += kOuter) {
    const int w = min(kOuter, m - j0);
    int rc = PotrfBlockColumn(s, m, j0, w, dH, ldh, d_info);
    if (rc != 0) return rc;
    const int rows = m - j0 - w;
    if (rows > 0) {
      // A22 -= L21 L21^T with K = w (lower tiles only)
      const double* L21 = dH + (long)j0 * ldh + (j0 + w);
      double* A22 = dH + (long)(j0 + w) * ldh + (j0 + w);
      rc = Dgemm(s, false, true, rows, rows, w, -1.0, L21, ldh, 0, L21, ldh, 0, 1.0, A22, ldh, 0, 1, true);
      if (rc != 0) return rc;
    }
  }
  return LaunchStatus();
}

// ---- pieces of the same factorisation for the distributed driver (host/distributed_cholesky.cc) ----
int cxb_potrf_max_panel(void) { return kOuter; }

int cxb_potrf_begin(void* stream, int* d_info) {
  CountLaunch(); ResetInfoKernel<<<1, 1, 0, AsStream(stream)>>>(d_info);
  return LaunchStatus();
}

int cxb_potrf_panel(void* stream, int m, int j0, int w, double* dH, long ldh, int* d_info) {
  if (m <= 0 || j0 < 0 || w <= 0 || w > kOuter || j0 + w > m) return -1;
  return PotrfBlockColumn(AsStream(stream), m, j0, w, dH, ldh, d_info);
}

// Partial factorisation of a front: `rows` x `cols` lower trapezoid (rows >= cols), the first `cols`
// columns are factored (L11 on top, L21 = A21 L11^{-T} below); trailing updates stay inside those
// columns. d_info is NOT reset (a chain of fronts shares one flag; once set, later fronts are no-ops).
int cxb_potrf_partial(void* stream, int rows, int cols, double* dF, long ld, int* d_info) {
  cudaStream_t s = AsStream(stream);
  if (rows < cols || cols < 0) return -1;
  for (int j0 = 0; j0 < cols; j0 += kOuter) {
    const int w = min(kOuter, cols - j0);
    int rc = PotrfBlockColumn(s, rows, j0, w, dF, ld, d_info);
    if (rc != 0) return rc;
    const int rest = cols - j0 - w;
    if (rest > 0) {
      const double* L21 = dF + (long)j0 * ld + (j0 + w);
      rc = Dgemm(s, false, true, rows - j0 - w, rest, w, -1.0, L21, ld, 0, L21, ld, 0, 1.0,
                 dF + (long)(j0 + w) * ld + (j0 + w), ld, 0, 1, true);
      if (rc != 0) return rc;
    }
  }
  return LaunchStatus();
}

// One sweep with an m x m lower-triangular block: transposed == 0: x <- L^{-1} x, else x <- L^{-T} x.
int cxb_trsv_lower(void* stream, int m, const double* dL, long ldl, double* dx, int transposed) {
  cudaStream_t s = AsStream(stream);
  if (m <= 0) return 0;
  ConfigureOnce();
  const int nblk = (m + kNB - 1) / kNB;
  // out-of-place sweep into a sentinel-filled scratch vector (+ the ticket behind it), copied back
  double* Z = nullptr;
  if (cudaMallocAsync(&Z, sizeof(double) * ((size_t)m + 2), s) != cudaSuccess) return (int)cudaErrorMemoryAllocation;
  int* ticket = reinterpret_cast<int*>(Z + m);
  CountLaunch(); WaveInitKernel<<<(m + 255) / 256, 256, 0, s>>>(Z, m, ticket, 1);
  CountLaunch();
  if (transposed) {
    TrsvBwdPollKernel<<<nblk, 512, kWaveSmem, s>>>(m, dL, ldl, dx, Z, ticket);
  } else {
    TrsvFwdPollKernel<<<nblk, 512, kWaveSmem, s>>>(m, dL, ldl, dx, Z, ticket);
  }
  cudaMemcpyAsync(dx, Z, sizeof(double) * (size_t)m, cudaMemcpyDeviceToDevice, s);
  cudaFreeAsync(Z, s);
  return LaunchStatus();
}

int cxb_scatter_lower_indexed(void* stream, int n, const double* dG, long ldg, const long* d_idx, double sign,
                              double* d_dst) {
  if (n <= 0) return 0;
  dim3 grid((n + 127) / 128, n);
  CountLaunch(); ScatterLowerIndexedKernel<<<grid, 128, 0, AsStream(stream)>>>(n, dG, ldg, d_idx, sign, d_dst);
  return LaunchStatus();
}

int cxb_front_forward(void* stream, int p, int sk, const double* dL21, long ld, const double* d_xk,
                      const int* d_sep, double* d_x) {
  if (p <= 0 || sk <= 0) return 0;
  CountLaunch(); FrontForwardKernel<<<(p + 7) / 8, 256, 0, AsStream(stream)>>>(p, sk, dL21, ld, d_xk, d_sep, d_x);
  return LaunchStatus();
}

int cxb_front_backward(void* stream, int p, int sk, const double* dL21, long ld, double* d_xk,
                       const int* d_sep, const double* d_x) {
  if (p <= 0 || sk <= 0) return 0;
  CountLaunch(); FrontBackwardKernel<<<(sk + 7) / 8, 256, 0, AsStream(stream)>>>(p, sk, dL21, ld, d_xk, d_sep, d_x);
  return LaunchStatus();
}

// X <- L^{-T} S L^{-1} X; signs == nullptr means S = I (plain Cholesky solve).
static int PotrsLowerImpl(cudaStream_t s, int m, const double* dL, long ldl, double* dX, long ldx, int nrhs,
                          const double* signs) {
  if (m <= 0 || nrhs <= 0) return 0;
  if (nrhs > kMaxRhs) return -1;
  ConfigureOnce();
  const int nblk = (m + kNB - 1) / kNB;
  // forward: dX (b) -> Z (z); backward: Z -> dX. Both outputs are sentinel-filled right before their sweep.
  const size_t mz = (size_t)m * nrhs;
  double* Z = nullptr;
  if (cudaMallocAsync(&Z, sizeof(double) * (mz + (size_t)nrhs + 1), s) != cudaSuccess) return (int)cudaErrorMemoryAllocation;
  int* tickets = reinterpret_cast<int*>(Z + mz);  // 2 * nrhs ints
  CountLaunch(); WaveInitKernel<<<(unsigned)((std::max<size_t>(mz, 2 * (size_t)nrhs) + 255) / 256), 256, 0, s>>>(Z, (long)mz, tickets, 2 * nrhs);
  for (int k = 0; k < nrhs; k++) {
    CountLaunch(); TrsvFwdPollKernel<<<nblk, 512, kWaveSmem, s>>>(m, dL, ldl, dX + (long)k * ldx, Z + (size_t)k * m, tickets + 2 * k);
  }
  if (signs) {
    CountLaunch(); ApplySignsKernel<<<(m + 255) / 256, 256, 0, s>>>(m, nrhs, signs, Z, m);
  }
  for (int k = 0; k < nrhs; k++) {
    CountLaunch(); WaveInitKernel<<<(m + 255) / 256, 256, 0, s>>>(dX + (long)k * ldx, m, nullptr, 0);
    CountLaunch(); TrsvBwdPollKernel<<<nblk, 512, kWaveSmem, s>>>(m, dL, ldl, Z + (size_t)k * m, dX + (long)k * ldx, tickets + 2 * k + 1);
  }
  cudaFreeAsync(Z, s);
  return LaunchStatus();
}

int cxb_potrs_lower(void* stream, int m, const double* dL, long ldl, double* dX, long ldx, int nrhs) {
  return PotrsLowerImpl(AsStream(stream), m, dL, ldl, dX, ldx, nrhs, nullptr);
}

size_t cxb_ldlt_worksize(int N) { return (size_t)N * kNB + (size_t)N; }

int cxb_sym_permute_lower(void* stream, int N, const double* dK, long ldk, const int* d_perm, double* dKp,
                          long ldp) {
  if (N <= 0) return 0;
  dim3 grid((N + 127) / 128, N);
  CountLaunch(); SymPermuteLowerKernel<<<grid, 128, 0, AsStream(stream)>>>(N, dK, ldk, d_perm, dKp, ldp);
  return LaunchStatus();
}

int cxb_ldlt_lower(void* stream, int N, double* dK, long ldk, double* d_signs, double* d_work, int* d_info) {
  cudaStream_t s = AsStream(stream);
  if (N <= 0) return 0;
  ConfigureOnce();
  CountLaunch(); ResetInfo2Kernel<<<1, 1, 0, s>>>(d_info);
  for (int i0 = 0; i0 < N; i0 += kNB) {
    const int nb = min(kNB, N - i0);
    double* Kii = dK + (long)i0 * ldk + i0;
    CountLaunch(); LdltDiagKernel<<<1, 512, kDiagSmem, s>>>(nb, Kii, ldk, i0, d_info, d_signs);
    const int rows = N - i0 - nb;
    if (rows <= 0) continue;
    double* A21 = Kii + nb;
    // d_info[0] stays 0 in signed mode, so the panel kernel's early-out never triggers
    CountLaunch(); TrsmPanelKernel<<<(rows + kNB - 1) / kNB, kNB, kTrsmSmem, s>>>(nb, Kii, ldk, A21, rows, d_info);
    dim3 grid((rows + 127) / 128, nb);
    CountLaunch(); SignedPanelKernel<<<grid, 128, 0, s>>>(rows, nb, A21, ldk, d_signs + i0, d_work);
    const int rc = DgemmEx(s, -1, 1, false, true, rows, rows, nb, -1.0, d_work, rows, 0, A21, ldk, 0, 1.0,
                           dK + (long)(i0 + nb) * ldk + (i0 + nb), ldk, 0, 1, true, false, 0);
    if (rc != 0) return rc;
  }
  return LaunchStatus();
}

// ---- LDL^T over fronts (multifrontal solver with equality multipliers) ---------------------------------
// Signed factorisation of the first `cols` columns of a rows x cols lower trapezoid (rows >= cols): on top
// L11 with F11 = L11 S L11^T, below G = F21 L11^{-T} S, so that the front is [L11; G] S [L11; G]^T and the Schur
// complement of the rows below is F22 - G S G^T. Trailing updates stay inside the `cols` columns. d_signs: cols
// entries (+-1); d_work: rows * 128 doubles; d_info[1] reports regularised pivots and is NOT reset here.
int cxb_ldlt_partial(void* stream, int rows, int cols, double* dF, long ld, double* d_signs, double* d_work,
                     int* d_info) {
  cudaStream_t s = AsStream(stream);
  if (rows < cols || cols < 0) return -1;
  if (cols == 0) return 0;
  ConfigureOnce();
  for (int i0 = 0; i0 < cols; i0 += kNB) {
    const int nb = min(kNB, cols - i0);
    double* Kii = dF + (long)i0 * ld + i0;
    CountLaunch(); LdltDiagKernel<<<1, 512, kDiagSmem, s>>>(nb, Kii, ld, i0, d_info, d_signs);
    const int below = rows - i0 - nb;
    if (below <= 0) continue;
    double* A21 = Kii + nb;
    CountLaunch(); TrsmPanelKernel<<<(below + kNB - 1) / kNB, kNB, kTrsmSmem, s>>>(nb, Kii, ld, A21, below, d_info);
    dim3 grid((below + 127) / 128, nb);
    CountLaunch(); SignedPanelKernel<<<grid, 128, 0, s>>>(below, nb, A21, ld, d_signs + i0, d_work);
    const int rest = cols - i0 - nb;  // columns of the front still to be updated
    if (rest > 0) {
      const int rc = DgemmEx(s, -1, 1, false, true, below, rest, nb, -1.0, d_work, below, 0, A21, ld, 0, 1.0,
                             dF + (long)(i0 + nb) * ld + (i0 + nb), ld, 0, 1, true, false, 0);
      if (rc != 0) return rc;
    }
  }
  return LaunchStatus();
}

int cxb_ldlt_begin(void* stream, int* d_info) {
  CountLaunch(); ResetInfo2Kernel<<<1, 1, 0, AsStream(stream)>>>(d_info);
  return LaunchStatus();
}

int cxb_front_permute(void* stream, int rows, int s_cols, const double* dF, long ld, const int* d_perm, double* dOut,
                      long ldo) {
  if (rows <= 0 || s_cols <= 0) return 0;
  dim3 grid((rows + 127) / 128, s_cols);
  CountLaunch(); FrontPermuteKernel<<<grid, 128, 0, AsStream(stream)>>>(rows, s_cols, dF, ld, d_perm, dOut, ldo);
  return LaunchStatus();
}

int cxb_scale_columns(void* stream, int rows, int cols, const double* dA, long lda, const double* d_signs,
                      double* dOut, long ldo) {
  if (rows <= 0 || cols <= 0) return 0;
  dim3 grid((rows + 127) / 128, cols);
  CountLaunch(); ScaleColumnsKernel<<<grid, 128, 0, AsStream(stream)>>>(rows, cols, dA, lda, d_signs, dOut, ldo);
  return LaunchStatus();
}

// out[i] = in[perm[i]] (scatter == 0) or out[perm[i]] = in[i] (scatter != 0)
int cxb_permute_vec(void* stream, int N, const int* d_perm, const double* d_in, double* d_out, int scatter) {
  if (N <= 0) return 0;
  CountLaunch(); PermuteVecKernel<<<(N + 255) / 256, 256, 0, AsStream(stream)>>>(N, d_perm, d_in, d_out, scatter);
  return LaunchStatus();
}

// x[i] *= signs[i]
int cxb_apply_signs(void* stream, int N, const double* d_signs, double* dx) {
  if (N <= 0) return 0;
  CountLaunch(); ApplySignsKernel<<<(N + 255) / 256, 256, 0, AsStream(stream)>>>(N, 1, d_signs, dx, N);
  return LaunchStatus();
}

int cxb_ldlt_solve(void* stream, int N, const double* dL, long ldl, const double* d_signs,
                   const int* d_perm, double* dx, double* d_tmp) {
  cudaStream_t s = AsStream(stream);
  if (N <= 0) return 0;
  CountLaunch(); PermuteVecKernel<<<(N + 255) / 256, 256, 0, s>>>(N, d_perm, dx, d_tmp, 0);
  const int rc = PotrsLowerImpl(s, N, dL, ldl, d_tmp, N, 1, d_signs);
  if (rc != 0) return rc;
  CountLaunch(); PermuteVecKernel<<<(N + 255) / 256, 256, 0, s>>>(N, d_perm, d_tmp, dx, 1);
  return LaunchStatus();
}

}  // extern "C"

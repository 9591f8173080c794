// Small cones, batched: one CTA per program of a batch; all per-problem arithmetic lives in
// small_cone_math.cuh (LP cone, second-order cone, small dense LMI block, small dense KKT system).
// This file only maps blockIdx.x to the program, carves shared memory and exports the C entry
// points declared in include/conex_b200_device.h.
#include "common.cuh"
#include "device_api.h"
#include "small_cone_math.cuh"
#include "small_psd_mma.cuh"
#include "team.cuh"

namespace cxb {
namespace {

constexpr int kThreads = 128;

__host__ __device__ inline long Align4(long n) { return (n + 3) & ~3L; }

struct ConeArgs {
  int type, n, m;
  int y_offset;  // in the padding after m: the struct keeps its size
  const double* data;
  long data_stride;
  double* state;
  long state_stride;
  double* work;
  long work_stride;
  const double* packed;
  long packed_stride;
};

static_assert(offsetof(cxb_small_cone, data) == 16 && sizeof(cxb_small_cone) == 80,
              "cxb_small_cone.y_offset must stay in the padding after m");

ConeArgs Convert(const cxb_small_cone* c) {
  return ConeArgs{c->type, c->n, c->m, c->y_offset, c->data, c->data_stride, c->state, c->state_stride, c->work,
                  c->work_stride, c->type == CXB_CONE_PSD ? c->packed : nullptr, c->packed_stride};
}

// Shared memory (doubles) needed by the PSD paths: 6 n^2 matrices + Lanczos vectors + slack + the scratch of the
// multi-section eigenvalue brackets.
size_t PsdSmemDoubles(int n) { return 6 * (size_t)n * n + 8 * (size_t)n + 64 + 2 * small::kSections + 16; }
// Second-order cones keep their scratch (o (m + 2) doubles: w^{1/2} and the scaled operator) in shared memory
// instead of the global `work` area: every use of it is local to one call.
// (Cones too large for that — more than kStagedLimit doubles — keep the global paths.)
constexpr long kStagedLimit = 12 * 1024;  // 96 KB
__host__ __device__ inline long SocScratchDoubles(int n, int m) { return (long)(n + 1) * (m + 2) + 4 * (long)(n + 1); }
// PsdEigen / PsdPrepare only touch sW | sS | sWS and the Lanczos vectors: 3 n^2 matrices instead of the 6 of the
// exponential map, so twice as many of their (latency-bound) CTAs fit on an SM.
size_t PsdSpectralSmemDoubles(int n) { return 3 * (size_t)n * n + 8 * (size_t)n + 64 + 2 * small::kSections + 16; }
size_t SmemBytes(const ConeArgs& c) {
  if (c.type == CXB_CONE_SOC) {
    const long need = SocScratchDoubles(c.n, c.m);
    return sizeof(double) * (64 + (need <= kStagedLimit ? need : 0));
  }
  return sizeof(double) * (64 + (c.type == CXB_CONE_PSD ? PsdSmemDoubles(c.n) : 0));
}
size_t SpectralSmemBytes(const ConeArgs& c) {
  if (c.type == CXB_CONE_PSD) return sizeof(double) * (64 + PsdSpectralSmemDoubles(c.n));
  return SmemBytes(c);
}
size_t SchurSmemBytes(const ConeArgs& c) {
  if (c.type == CXB_CONE_SOC) return SmemBytes(c);
  if (c.type == CXB_CONE_LP) {
    const long need = small::LpSchurSmemDoubles(c.n, c.m);
    return sizeof(double) * (64 + (need <= kStagedLimit ? need : 0));
  }
  return sizeof(double) * (64 + (size_t)small::PsdSchurSmemDoubles(c.n, c.m, kThreads));
}
// The scratch of a second-order cone: shared memory when the launch reserved it, else the global work area.
__device__ __forceinline__ double* SocScratch(const ConeArgs& c, long per, double* base, double* work) {
  return per >= 64 + SocScratchDoubles(c.n, c.m) ? base + 64 : work;
}

// Two thread layouts for the same phase-structured math (small_cone_math.cuh):
//   WARP == false: one CTA of kThreads threads per program (DeviceTeam, block barriers between phases);
//   WARP == true : one WARP per program, several programs per CTA (WarpTeam: __syncwarp + shuffles). Default only
//                  for the kernel that is one dependent chain (the triangular solves of the small KKT systems):
//                  everywhere else it measured slower, because the shared memory of a problem, not its threads,
//                  bounds how many problems an SM holds (cxb_set_small_team_mode, DESIGN.md 3.2).
// `per` = doubles of dynamic shared memory per program.
template <bool WARP>
struct TeamOf {
  using type = DeviceTeam;
  static __device__ __forceinline__ DeviceTeam Make(double* base) { return DeviceTeam(base); }
};
template <>
struct TeamOf<true> {
  using type = WarpTeam;
  static __device__ __forceinline__ WarpTeam Make(double*) { return WarpTeam(); }
};
template <bool WARP>
__device__ __forceinline__ bool Slot(int batch, long per, double* sm, const int* active, int* p, double** base) {
  if (WARP) {
    const int w = threadIdx.x >> 5;
    *p = blockIdx.x * (blockDim.x >> 5) + w;
    *base = sm + w * per;
  } else {
    *p = blockIdx.x;
    *base = sm;
  }
  return *p < batch && !(active && !active[*p]);
}

template <bool WARP>
__device__ __forceinline__ void SetIdentityBody(int batch, long per, const ConeArgs& c, const int* active) {
  extern __shared__ double sm[];
  int p;
  double* base;
  if (!Slot<WARP>(batch, per, sm, active, &p, &base)) return;
  auto t = TeamOf<WARP>::Make(base);
  double* st = c.state + p * c.state_stride;
  if (c.type == CXB_CONE_LP) {
    t.par(c.n, [&](int i) { st[i] = 1.0; });
  } else if (c.type == CXB_CONE_SOC) {
    small::SocSetIdentity(t, c.n + 1, st);
  } else {
    small::PsdSetIdentity(t, c.n, st);
  }
}

template <bool WARP>
__global__ void __launch_bounds__(kThreads) SchurKernel(int batch, long per, ConeArgs c, double* G, long ldg,
                                                        long gstride, double* AW, double* AQc, long vstride,
                                                        double* scal, long sstride, int accumulate,
                                                        const int* active) {
  extern __shared__ double sm[];
  int p;
  double* base;
  if (!Slot<WARP>(batch, per, sm, active, &p, &base)) return;
  auto t = TeamOf<WARP>::Make(base);
  const double* data = c.data + p * c.data_stride;
  double* st = c.state + p * c.state_stride;
  double* work = c.work ? c.work + p * c.work_stride : nullptr;
  const bool lp_staged = per >= 64 + small::LpSchurSmemDoubles(c.n, c.m);  // large LP cones: straight from global
  double* g = G + p * gstride;
  double* aw = AW + p * vstride;
  double* aq = AQc + p * vstride;
  double* sc = scal + p * sstride;
  const bool acc = accumulate != 0;
  if (c.type == CXB_CONE_LP) {
    small::LpSchur(t, c.n, c.m, data, st, g, ldg, aw, aq, sc, acc, lp_staged ? base + 64 : nullptr);
  } else if (c.type == CXB_CONE_SOC) {
    small::SocSchur(t, c.n + 1, c.m, data, st, SocScratch(c, per, base, work), g, ldg, aw, aq, sc, acc);
  } else {
    small::PsdSchur(t, c.n, c.m, data, st, work, base + 64, g, ldg, aw, aq, sc, acc);
  }
}

// Dense LMI blocks of order n <= 32, n % 4 == 0: the DMMA kernel of small_psd_mma.cuh (one CTA of 16 warps per
// program, scaled matrices kept in shared memory).
template <int NT>
__global__ void __launch_bounds__(psdmma::kThreads, 1) PsdSchurMmaKernel(ConeArgs c, double* G, long ldg, long gstride,
                                                                       double* AW, double* AQc, long vstride,
                                                                       double* scal, long sstride, int accumulate,
                                                                       const int* active) {
  extern __shared__ __align__(16) double sm[];
  const int p = blockIdx.x;
  if (active && !active[p]) return;
  double* work = c.work + p * c.work_stride;  // holds the factor image written by PsdFactorKernel
  psdmma::PsdSchurMma<NT>(c.n, c.m, c.data + p * c.data_stride, c.state + p * c.state_stride, work, work, sm,
                          G + p * gstride, ldg, AW + p * vstride, AQc + p * vstride, scal + p * sstride,
                          accumulate != 0);
}

template <int N4>
__global__ void __launch_bounds__(psdmma::kThreads2, 2) PsdSchurMma2Kernel(ConeArgs c, double* G, long ldg, long gstride,
                                                                         double* AW, double* AQc, long vstride,
                                                                         double* scal, long sstride, int accumulate,
                                                                         const int* active) {
  extern __shared__ __align__(16) double sm[];
  const int p = blockIdx.x;
  if (active && !active[p]) return;
  double* work = c.work + p * c.work_stride;
  psdmma::PsdSchurMma2<N4>(c.m, c.data + p * c.data_stride, c.state + p * c.state_stride, work, work, sm,
                           G + p * gstride, ldg, AW + p * vstride, AQc + p * vstride, scal + p * sstride,
                           accumulate != 0);
}

// L = chol(W) of every program's block, one warp per program, into the head of the program's `work` area.
__global__ void __launch_bounds__(128) PsdFactorKernel(int batch, ConeArgs c, const int* active) {
  extern __shared__ double sm[];
  const int w = threadIdx.x >> 5;
  const int p = blockIdx.x * 4 + w;
  if (p >= batch || (active && !active[p])) return;
  psdmma::PsdFactorWarp(c.n, c.state + p * c.state_stride, sm + (long)w * (psdmma::LImageDoubles(c.n) + 2),
                        c.work + p * c.work_stride);
}

template <bool WARP>
__device__ __forceinline__ void EigenBody(int batch, long per, const ConeArgs& c, const double* y, long ystride,
                                          double cw, const double* cw_p, double* out4, long ostride,
                                          const int* active) {
  extern __shared__ double sm[];
  int p;
  double* base;
  if (!Slot<WARP>(batch, per, sm, active, &p, &base)) return;
  auto t = TeamOf<WARP>::Make(base);
  const double* data = c.data + p * c.data_stride;
  double* st = c.state + p * c.state_stride;
  double* work = c.work ? c.work + p * c.work_stride : nullptr;
  const double* yp = y + p * ystride + c.y_offset;
  const double k = cw_p ? cw_p[p] : cw;
  double* out = out4 + p * ostride;
  if (c.type == CXB_CONE_LP) {
    const long np = Align4(c.n);
    small::LpEigen(t, c.n, c.m, data, yp, k, st, st + np, st + 2 * np, out);
  } else if (c.type == CXB_CONE_SOC) {
    small::SocEigen(t, c.n + 1, c.m, data, yp, k, st, SocScratch(c, per, base, work), out);
  } else {
    const long nnp = Align4((long)c.n * c.n);
    small::PsdEigen(t, c.n, c.m, data, yp, k, st, st + nnp, st + 2 * nnp, base + 64, out,
                    c.packed ? c.packed + p * c.packed_stride : nullptr);
  }
}

template <bool WARP>
__device__ __forceinline__ void PrepareBody(int batch, long per, const ConeArgs& c, const double* y, long ystride,
                                            int affine, double cw, const double* cw_p, double ew, double* out2,
                                            long ostride, const int* active) {
  extern __shared__ double sm[];
  int p;
  double* base;
  if (!Slot<WARP>(batch, per, sm, active, &p, &base)) return;
  auto t = TeamOf<WARP>::Make(base);
  const double* data = c.data + p * c.data_stride;
  double* st = c.state + p * c.state_stride;
  double* work = c.work ? c.work + p * c.work_stride : nullptr;
  const double* yp = y + p * ystride + c.y_offset;
  const double k = cw_p ? cw_p[p] : cw;
  double* out = out2 + p * ostride;
  if (c.type == CXB_CONE_LP) {
    const long np = Align4(c.n);
    small::LpPrepare(t, c.n, c.m, data, yp, affine != 0, k, ew, st, st + np, st + 2 * np, out);
  } else if (c.type == CXB_CONE_SOC) {
    const long op = Align4(c.n + 1);
    small::SocPrepare(t, c.n + 1, c.m, data, yp, k, st, st + op, SocScratch(c, per, base, work), out);
  } else {
    const long nnp = Align4((long)c.n * c.n);
    small::PsdPrepare(t, c.n, c.m, data, yp, affine != 0, k, ew, st, st + nnp, st + 2 * nnp, base + 64, out,
                      c.packed ? c.packed + p * c.packed_stride : nullptr);
  }
}

template <bool WARP>
__device__ __forceinline__ void TakeStepBody(int batch, long per, const ConeArgs& c, double step,
                                             const double* step_p, double ew, int* info, const int* active) {
  extern __shared__ double sm[];
  int p;
  double* base;
  if (!Slot<WARP>(batch, per, sm, active, &p, &base)) return;
  auto t = TeamOf<WARP>::Make(base);
  double* st = c.state + p * c.state_stride;
  double* work = c.work ? c.work + p * c.work_stride : nullptr;
  const double s = step_p ? step_p[p] : step;
  if (c.type == CXB_CONE_LP) {
    const long np = Align4(c.n);
    small::LpTakeStep(t, c.n, s, st, st + 2 * np);
  } else if (c.type == CXB_CONE_SOC) {
    const long op = Align4(c.n + 1);
    small::SocTakeStep(t, c.n + 1, s, st, st + op, SocScratch(c, per, base, work));
  } else {
    const long nnp = Align4((long)c.n * c.n);
    small::PsdTakeStep(t, c.n, s, ew, st, st + 2 * nnp, base + 64, info + p);
  }
}


// One launch per cone (any layout) and one launch for a list of cones (CTA layout, blockIdx.y = cone): the lock step of
// a batch of multi-cone programs runs the same operation on every cone, and launched one after the other the cones'
// dependent chains (Lanczos, Gaussian elimination) serialise while most of the SMs idle when the batch is small.
constexpr int kMaxFused = 8;
struct ConeList {
  ConeArgs c[kMaxFused];
};

template <bool WARP>
__global__ void __launch_bounds__(kThreads) SetIdentityKernel(int batch, long per, ConeArgs c, const int* active) {
  SetIdentityBody<WARP>(batch, per, c, active);
}
__global__ void __launch_bounds__(kThreads) SetIdentityMultiKernel(int batch, long per, ConeList l, const int* active) {
  SetIdentityBody<false>(batch, per, l.c[blockIdx.y], active);
}
template <bool WARP>
__global__ void __launch_bounds__(kThreads) EigenKernel(int batch, long per, ConeArgs c, const double* y, long ystride,
                                                        double cw, const double* cw_p, double* out4,
                                                        long ostride, const int* active) {
  EigenBody<WARP>(batch, per, c, y, ystride, cw, cw_p, out4, ostride, active);
}
__global__ void __launch_bounds__(kThreads, 8) EigenMultiKernel(int batch, long per, ConeList l, const double* y,
                                                             long ystride, double cw, const double* cw_p, double* out4,
                                                             long ostride, const int* active) {
  EigenBody<false>(batch, per, l.c[blockIdx.y], y, ystride, cw, cw_p, out4 + 4 * blockIdx.y, ostride, active);
}
template <bool WARP>
__global__ void __launch_bounds__(kThreads) PrepareKernel(int batch, long per, ConeArgs c, const double* y,
                                                          long ystride, int affine, double cw, const double* cw_p,
                                                          double ew, double* out2, long ostride,
                                                          const int* active) {
  PrepareBody<WARP>(batch, per, c, y, ystride, affine, cw, cw_p, ew, out2, ostride, active);
}
__global__ void __launch_bounds__(kThreads, 8) PrepareMultiKernel(int batch, long per, ConeList l, const double* y,
                                                               long ystride, int affine, double cw, const double* cw_p,
                                                               double ew, double* out2, long ostride,
                                                               const int* active) {
  PrepareBody<false>(batch, per, l.c[blockIdx.y], y, ystride, affine, cw, cw_p, ew, out2 + 4 * blockIdx.y, ostride,
                     active);
}
template <bool WARP>
__global__ void __launch_bounds__(kThreads) TakeStepKernel(int batch, long per, ConeArgs c, double step,
                                                           const double* step_p, double ew, int* info,
                                                           const int* active) {
  TakeStepBody<WARP>(batch, per, c, step, step_p, ew, info, active);
}
__global__ void __launch_bounds__(kThreads) TakeStepMultiKernel(int batch, long per, ConeList l, double step,
                                                                const double* step_p, double ew, int* info,
                                                                const int* active) {
  TakeStepBody<false>(batch, per, l.c[blockIdx.y], step, step_p, ew, info, active);
}

// Lower triangles of the matrices [first, first + count) of a PSD cone, one CTA per program; flags matrices that are
// not symmetric.
__global__ void __launch_bounds__(kThreads) PackSymmetricKernel(ConeArgs c, int first, int count, double* packed,
                                                               long packed_stride, int* asymmetric) {
  const int p = blockIdx.x;
  const int n = c.n, kp = n * (n + 1) / 2;
  const double* data = c.data + p * c.data_stride + (long)first * n * n;
  double* out = packed + p * packed_stride + (long)first * kp;
  bool bad = false;
  for (int e = threadIdx.x; e < count * n * n; e += blockDim.x) {
    const int j = e / (n * n), q = e - j * n * n;
    const int col = q / n, row = q - col * n;
    if (row < col) continue;
    const double v = data[e];
    bad = bad || !(v == data[(long)j * n * n + (long)row * n + col]);
    out[(long)j * kp + col * n - col * (col - 1) / 2 + (row - col)] = v;
  }
  if (bad) *asymmetric = 1;
}

template <bool WARP>
__global__ void __launch_bounds__(kThreads) PotrfKernel(int batch, long per, int N, double* H, long ldh, long hstride,
                                                        int* info, const int* active) {
  extern __shared__ double sm[];
  int p;
  double* base;
  if (!Slot<WARP>(batch, per, sm, active, &p, &base)) return;
  auto t = TeamOf<WARP>::Make(base);
  small::SmallPotrf(t, N, H + p * hstride, ldh, base + 64, info + p);
}

template <bool WARP>
__global__ void __launch_bounds__(kThreads) PotrsKernel(int batch, long per, int N, const double* L, long ldl,
                                                        long lstride, double* X, long xstride, const int* active) {
  extern __shared__ double sm[];
  int p;
  double* base;
  if (!Slot<WARP>(batch, per, sm, active, &p, &base)) return;
  auto t = TeamOf<WARP>::Make(base);
  small::SmallPotrs(t, N, L + p * lstride, ldl, X + p * xstride, base + 64);
}

// Shared memory (doubles) of the regularised LDL^T: the permuted copy, the |diagonal| and the pivot order (ints).
__host__ __device__ inline long LdltSmemDoubles(int N) { return (long)N * N + N + (N + 1) / 2; }

template <bool WARP>
__global__ void __launch_bounds__(kThreads) LdltKernel(int batch, long per, int N, const double* K, long ldk,
                                                       long kstride, double* L, long ldl, long lstride, int* perm,
                                                       long pstride, double* signs, long sstride, int* info,
                                                       const int* active) {
  extern __shared__ double sm[];
  int p;
  double* base;
  if (!Slot<WARP>(batch, per, sm, active, &p, &base)) return;
  auto t = TeamOf<WARP>::Make(base);
  double* sH = base + 64;
  const int regularised = small::SmallLdlt(t, N, K + p * kstride, ldk, L + p * lstride, ldl, perm + p * pstride,
                                           signs + p * sstride, sH, sH + (long)N * N,
                                           reinterpret_cast<int*>(sH + (long)N * N + N));
  // written here rather than inside SmallLdlt: a pointer live across the whole factorisation was spilled
  t.single([&]() { info[p] = regularised; });
}

template <bool WARP>
__global__ void __launch_bounds__(kThreads) LdltSolveKernel(int batch, long per, int N, const double* L, long ldl,
                                                            long lstride, const int* perm, long pstride,
                                                            const double* signs, long sstride, double* X,
                                                            long xstride, const int* active) {
  extern __shared__ double sm[];
  int p;
  double* base;
  if (!Slot<WARP>(batch, per, sm, active, &p, &base)) return;
  auto t = TeamOf<WARP>::Make(base);
  small::SmallLdltSolve(t, N, L + p * lstride, ldl, perm + p * pstride, signs + p * sstride, X + p * xstride,
                        base + 64);
}

// ---- KKT systems larger than shared memory: small::BlockedPotrf / BlockedLdlt, one CTA of kThreads per program ----
// The trailing update A22 -= L21 S L21^T of a block column on the FP64 tensor cores: the lower 32 x 32 tiles of A22
// go round the warps; per tile the warp stages its two operand panels (kb <= 32 columns each) in its own shared
// memory, -L21 rows of the tile's row block and S L21 rows of its column block, k-major with a pitch of 4 (mod 16)
// so that the fragment loads are conflict free, and accumulates on top of the tile read from global memory.
constexpr int kKktTile = small::kKktNb;
constexpr int kKktOpPitch = 36;
constexpr long kKktStageDoubles = 2L * kKktTile * kKktOpPitch;  // per warp
struct KktTrailingUpdateMma {
  double* stage;  // kThreads / 32 * kKktStageDoubles doubles of shared memory
  __device__ void operator()(DeviceTeam& t, double* A, long ld, int k0, int kb, int t0, int R, const double* s) const {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int gid = lane >> 2, tig = lane & 3;
    double* sa = stage + warp * kKktStageDoubles;  // sa[k * pitch + r] = -L21(r0 + r, k)
    double* sb = sa + kKktTile * kKktOpPitch;      // sb[k * pitch + c] = s_k L21(c0 + c, k)
    const int nt = (R + kKktTile - 1) / kKktTile;
    const int k4 = (kb + 3) & ~3;
    const double* L21 = A + (long)k0 * ld + t0;
    double* A22 = A + (long)t0 * ld + t0;
    for (int w = warp; w < nt * (nt + 1) / 2; w += nwarps) {
      int ti = (int)((sqrt(8.0 * w + 1.0) - 1.0) * 0.5);  // row-major order of the lower tiles: w -> (ti >= tj)
      while ((ti + 1) * (ti + 2) / 2 <= w) ti++;
      while (ti * (ti + 1) / 2 > w) ti--;
      const int tj = w - ti * (ti + 1) / 2;
      const int r0 = ti * kKktTile, c0 = tj * kKktTile;
      for (int e = lane; e < k4 * kKktTile; e += 32) {
        const int k = e / kKktTile, r = e % kKktTile;
        const bool in = k < kb;
        sa[k * kKktOpPitch + r] = (in && r0 + r < R) ? -L21[(long)k * ld + r0 + r] : 0.0;
        sb[k * kKktOpPitch + r] = (in && c0 + r < R) ? s[k] * L21[(long)k * ld + c0 + r] : 0.0;
      }
      __syncwarp();
      // acc[x][y] = A22(r0 + 8 x + gid, c0 + 8 y + 2 tig + {0, 1}); entries outside A22 stay zero, entries above its
      // diagonal (diagonal tiles) are not read
      double acc[4][4][2];
#pragma unroll
      for (int x = 0; x < 4; x++)
#pragma unroll
        for (int y = 0; y < 4; y++)
#pragma unroll
          for (int h = 0; h < 2; h++) {
            const int r = r0 + 8 * x + gid, c = c0 + 8 * y + 2 * tig + h;
            acc[x][y][h] = (r < R && c <= r) ? A22[(long)c * ld + r] : 0.0;
          }
      const bool diag = ti == tj;
      for (int k = 0; k < k4; k += 4) {
        double a[4], b[4];
#pragma unroll
        for (int x = 0; x < 4; x++) a[x] = sa[(k + tig) * kKktOpPitch + 8 * x + gid];
#pragma unroll
        for (int y = 0; y < 4; y++) b[y] = sb[(k + tig) * kKktOpPitch + 8 * y + gid];
#pragma unroll
        for (int x = 0; x < 4; x++)
#pragma unroll
          for (int y = 0; y < 4; y++)
            if (!diag || y <= x) Dmma884(acc[x][y][0], acc[x][y][1], a[x], b[y]);
      }
#pragma unroll
      for (int x = 0; x < 4; x++)
#pragma unroll
        for (int y = 0; y < 4; y++)
#pragma unroll
          for (int h = 0; h < 2; h++) {
            const int r = r0 + 8 * x + gid, c = c0 + 8 * y + 2 * tig + h;
            if (r < R && c <= r) A22[(long)c * ld + r] = acc[x][y][h];
          }
      __syncwarp();  // the next tile's staging overwrites sa / sb
    }
    __syncthreads();  // the next block column reads the updated trailing matrix
  }
};

// Dynamic shared memory (doubles) of the blocked kernels: reduction scratch, the diagonal block, the warps' operand
// stages and (LDL^T) the pivot order, N doubles and N ints.
__host__ __device__ inline long BlockedKktSmemDoubles(int N, bool ldlt) {
  return 64 + small::BlockedKktSmemDoubles() + (kThreads / 32) * kKktStageDoubles + (ldlt ? N + (N + 1) / 2 : 0);
}

__global__ void __launch_bounds__(kThreads) BlockedPotrfKernel(int N, double* H, long ldh, long hstride, int* info,
                                                               const int* active) {
  extern __shared__ double sm[];
  const int p = blockIdx.x;
  if (active && !active[p]) return;
  DeviceTeam t(sm);
  double* scratch = sm + 64;
  const KktTrailingUpdateMma update{scratch + small::BlockedKktSmemDoubles()};
  const int failed = small::BlockedPotrf(t, N, H + p * hstride, ldh, scratch, update);
  t.single([&]() { info[p] = failed; });
}

__global__ void __launch_bounds__(kThreads) BlockedLdltKernel(int N, const double* K, long ldk, long kstride, double* L,
                                                              long ldl, long lstride, int* perm, long pstride,
                                                              double* signs, long sstride, int* info,
                                                              const int* active) {
  extern __shared__ double sm[];
  const int p = blockIdx.x;
  if (active && !active[p]) return;
  DeviceTeam t(sm);
  double* scratch = sm + 64;
  double* stage = scratch + small::BlockedKktSmemDoubles();
  double* sd = stage + (kThreads / 32) * kKktStageDoubles;
  const KktTrailingUpdateMma update{stage};
  const int regularised = small::BlockedLdlt(t, N, K + p * kstride, ldk, L + p * lstride, ldl, perm + p * pstride,
                                             signs + p * sstride, scratch, sd, reinterpret_cast<int*>(sd + N), update);
  t.single([&]() { info[p] = regularised; });
}

// The y slices of the subset cones of a batch (cxb_small_gather): one CTA per program.
__global__ void __launch_bounds__(kThreads) GatherKernel(int count, const int* __restrict__ idx, double* y,
                                                         long ystride, long dst, const int* active) {
  const int p = blockIdx.x;
  if (active && !active[p]) return;
  double* yp = y + p * ystride;
  for (int i = threadIdx.x; i < count; i += blockDim.x) {
    const int v = idx[i];
    if (v >= 0) yp[dst + i] = yp[v];
  }
}

// The Schur blocks of the subset cones into H / AW / AQc / scal (cxb_small_scatter_schur): one CTA per program, the
// cones one after the other. Within a cone the targets are distinct (its variables are), so its entries are split
// over the threads without atomics.
__global__ void __launch_bounds__(kThreads) ScatterSchurKernel(int ncones, const int* __restrict__ cones,
                                                               const int* __restrict__ idx, const double* S,
                                                               long sstride, int m, double* H, long ldh, long hstride,
                                                               double* AW, double* AQc, long vstride, double* scal,
                                                               long scal_stride, int accumulate, const int* active) {
  const int p = blockIdx.x;
  if (active && !active[p]) return;
  double* h = H + p * hstride;
  double* aw = AW + p * vstride;
  double* aq = AQc + p * vstride;
  double* sc = scal + p * scal_stride;
  const double* s = S + p * sstride;
  if (!accumulate) {
    for (int e = threadIdx.x; e < m * m; e += blockDim.x) {
      const int j = e / m, i = e - j * m;
      h[i + (long)j * ldh] = 0;
    }
    for (int i = threadIdx.x; i < m; i += blockDim.x) aw[i] = aq[i] = 0;
    if (threadIdx.x == 0) sc[0] = sc[1] = 0;
    __syncthreads();
  }
  for (int k = 0; k < ncones; k++) {
    const int mk = cones[3 * k];
    const int* v = idx + cones[3 * k + 1];
    const double* g = s + cones[3 * k + 2];
    const long ld = Align4(mk);
    for (int e = threadIdx.x; e < mk * mk; e += blockDim.x) {
      const int j = e / mk, i = e - j * mk;
      if (i < j) continue;
      const int vi = v[i], vj = v[j];
      h[(vi > vj ? vi : vj) + (long)(vi > vj ? vj : vi) * ldh] += g[i + j * ld];
    }
    for (int i = threadIdx.x; i < mk; i += blockDim.x) {
      aw[v[i]] += g[ld * mk + i];
      aq[v[i]] += g[ld * (mk + 1) + i];
    }
    if (threadIdx.x == 0) {
      sc[0] += g[ld * (mk + 2)];
      sc[1] += g[ld * (mk + 2) + 1];
    }
    __syncthreads();  // the next cone may share targets with this one
  }
}

__global__ void LincombKernel(int n, const double* a, const double* x, long xs, const double* b,
                              const double* y, long ys, const double* c, const double* z, long zs,
                              double* out, long os, const int* active) {
  const int p = blockIdx.y;
  if (active && !active[p]) return;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double v = 0;
  if (a && x) v += a[p] * x[p * xs + i];
  if (b && y) v += b[p] * y[p * ys + i];
  if (c && z) v += c[p] * z[p * zs + i];
  out[p * os + i] = v;
}

__global__ void __launch_bounds__(kThreads) BatchedDotKernel(int n, const double* x, long xs,
                                                             const double* y, long ys, double* out,
                                                             long ostride) {
  __shared__ double scratch[40];
  const int p = blockIdx.x;
  double s = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s += x[p * xs + i] * y[p * ys + i];
  s = BlockSum(s, scratch);
  if (threadIdx.x == 0) out[p * ostride] = s;
}

constexpr size_t kMaxSmemBytes = 227 * 1024;  // dynamic shared memory of one CTA on sm_100

template <typename K>
int EnsureSmem(K kernel, size_t bytes) {
  if (bytes > kMaxSmemBytes) return -1;
  if (bytes > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return (int)e;
  }
  return 0;
}

// dense-LMI branch of cxb_small_schur (cxb_set_small_psd_mma): 2 = DMMA kernel, 8 warps per CTA, two CTAs per SM
// (default; falls back to 1 when its shared memory does not fit twice); 1 = DMMA kernel, 16 warps, whole operator in
// shared memory, one CTA per SM; 0 = the DFMA team kernel
int g_small_psd_mma = 2;
// cxb_set_small_team_mode: 2 (default) = one warp per program for the triangular solves of the small KKT systems only
// (the one kernel whose phases are all a single dependent chain), one CTA per program elsewhere; 1 = one warp per
// program everywhere; 0 = one CTA per program everywhere. Measured on C3 (profiles/r02_e_bench_c3_variants.txt): the
// warp layout is 1.8x faster for the solves and 1.3-1.5x SLOWER for the kernels that have real parallel phases.
int g_small_team_mode = 2;

bool ValidCone(const cxb_small_cone* c) {
  if (!c || c->n < 1 || c->m < 1 || c->y_offset < 0 || !c->data || !c->state) return false;
  if (c->type == CXB_CONE_LP) return true;
  if (c->type == CXB_CONE_SOC) return c->work != nullptr;
  if (c->type == CXB_CONE_PSD) return c->work != nullptr && c->n <= 64;
  return false;
}

}  // namespace
}  // namespace cxb

using namespace cxb;

extern "C" {

size_t cxb_small_state_size(int type, int n) {
  if (type == CXB_CONE_LP) return 3 * (size_t)Align4(n);
  if (type == CXB_CONE_SOC) return 2 * (size_t)Align4(n + 1);
  return 3 * (size_t)Align4((long)n * n);
}

size_t cxb_small_work_size(int type, int n, int m) {
  if (type == CXB_CONE_LP) return 0;
  if (type == CXB_CONE_SOC) return (size_t)(n + 1) * (m + 4);
  return (size_t)(m + 2) * n * n;
}

namespace {
// Launch geometry of the two layouts: `per` doubles of shared memory per program. Warp layout: as many programs
// per CTA (<= 4 warps) as fit in ~100 KB, so that at least two CTAs share an SM.
struct Geometry {
  bool warp;
  int grid, threads;
  long per;
  size_t smem;
};
// CTA size of the spectral kernels (cxb_small_eigen / cxb_small_prepare) in the CTA layout (cxb_set_small_cone_threads).
int g_spectral_threads = 64;  // measured on C3: 57.0 ms (64) / 57.6 (32) / 59.5 (128), profiles/r02_j_bench_c3_variants.txt
Geometry MakeGeometry(int batch, size_t per_program_bytes, bool chain_only = false, int threads = kThreads) {
  Geometry g;
  g.per = (long)(per_program_bytes / sizeof(double));
  // a single program (the LP / SOC plugins of CONEX_Maximize) keeps the whole CTA: its cones can be large
  g.warp = (g_small_team_mode == 1 || (g_small_team_mode == 2 && chain_only)) && batch >= 8;
  if (g.warp) {
    int w = (int)((100 * 1024) / (per_program_bytes > 0 ? per_program_bytes : 1));
    w = w < 1 ? 1 : (w > 4 ? 4 : w);
    g.threads = 32 * w;
    g.grid = (batch + w - 1) / w;
    g.smem = per_program_bytes * w;
  } else {
    g.threads = threads;
    g.grid = batch;
    g.smem = per_program_bytes;
  }
  return g;
}

// The cones [first, first + count) of a list as kernel arguments; *smem = the largest per-cone requirement.
extern "C++" template <class SmemOf>
bool MakeList(int count, const cxb_small_cone* cones, SmemOf smem_of, ConeList* list, size_t* smem) {
  *smem = 0;
  for (int k = 0; k < count; k++) {
    if (!ValidCone(cones + k)) return false;
    list->c[k] = Convert(cones + k);
    const size_t b = smem_of(list->c[k]);
    if (b > *smem) *smem = b;
  }
  return true;
}
// the fused launches use the CTA layout; with the warp layout forced everywhere the cones are launched one by one
int g_small_fused = 1;  // cxb_set_small_fused_launches: A/B switch
bool FusedLayout(int batch) { return g_small_fused && !(g_small_team_mode == 1 && batch >= 8); }
}  // namespace

int cxb_small_set_identity(void* stream, int batch, const cxb_small_cone* cone, const int* d_active) {
  if (batch <= 0) return 0;
  if (!ValidCone(cone)) return -1;
  const ConeArgs c = Convert(cone);
  const Geometry g = MakeGeometry(batch, sizeof(double) * 64);
  CountLaunch();
  if (g.warp) {
    SetIdentityKernel<true><<<g.grid, g.threads, g.smem, AsStream(stream)>>>(batch, g.per, c, d_active);
  } else {
    SetIdentityKernel<false><<<g.grid, g.threads, g.smem, AsStream(stream)>>>(batch, g.per, c, d_active);
  }
  return LaunchStatus();
}

int cxb_small_pack_symmetric_columns(void* stream, int batch, const cxb_small_cone* cone, int first, int count,
                                     double* d_packed, long packed_stride, int* d_asymmetric) {
  if (batch <= 0) return 0;
  if (!ValidCone(cone) || cone->type != CXB_CONE_PSD || !d_packed || !d_asymmetric) return -1;
  if (first < 0 || count < 1 || first + count > cone->m + 1) return -1;
  if (packed_stride < (long)(cone->m + 1) * (cone->n * (cone->n + 1) / 2)) return -1;
  ConeArgs c = Convert(cone);
  CountLaunch();
  PackSymmetricKernel<<<batch, kThreads, 0, AsStream(stream)>>>(c, first, count, d_packed, packed_stride,
                                                                d_asymmetric);
  return LaunchStatus();
}

int cxb_small_pack_symmetric(void* stream, int batch, const cxb_small_cone* cone, double* d_packed, long packed_stride,
                             int* d_asymmetric) {
  if (batch <= 0) return 0;
  if (!cone) return -1;
  return cxb_small_pack_symmetric_columns(stream, batch, cone, 0, cone->m + 1, d_packed, packed_stride, d_asymmetric);
}

int cxb_small_schur(void* stream, int batch, const cxb_small_cone* cone, double* dG, long ldg,
                    long gstride, double* dAW, double* dAQc, long vstride, double* d_scal, long sstride,
                    int accumulate, const int* d_active) {
  if (batch <= 0) return 0;
  if (!ValidCone(cone)) return -1;
  const ConeArgs c = Convert(cone);
  size_t mma_smem = 0;
  const bool aligned = (c.data_stride % 2) == 0 && (reinterpret_cast<uintptr_t>(c.data) & 15) == 0;
  const bool two_per_sm = g_small_psd_mma == 2 && c.type == CXB_CONE_PSD && aligned && psdmma::Supported2(c.n, c.m, &mma_smem);
  if (two_per_sm || (c.type == CXB_CONE_PSD && g_small_psd_mma && aligned && psdmma::Supported(c.n, c.m, &mma_smem))) {
    const int threads = two_per_sm ? psdmma::kThreads2 : psdmma::kThreads;
    auto launch = [&](auto kernel) -> int {
      int rc = EnsureSmem(kernel, mma_smem);
      if (rc) return rc;
      CountLaunch(); PsdFactorKernel<<<(batch + 3) / 4, 128, sizeof(double) * 4 * (psdmma::LImageDoubles(c.n) + 2),
                                       AsStream(stream)>>>(batch, c, d_active);
      CountLaunch(); kernel<<<batch, threads, mma_smem, AsStream(stream)>>>(
          c, dG, ldg, gstride, dAW, dAQc, vstride, d_scal, sstride, accumulate, d_active);
      return LaunchStatus();
    };
    const int nt = (c.n + 7) / 8;
    if (two_per_sm) {
      switch (c.n / 4) {  // Supported2: n = 4, 8, ..., 32
        case 1: return launch(PsdSchurMma2Kernel<1>);
        case 2: return launch(PsdSchurMma2Kernel<2>);
        case 3: return launch(PsdSchurMma2Kernel<3>);
        case 4: return launch(PsdSchurMma2Kernel<4>);
        case 5: return launch(PsdSchurMma2Kernel<5>);
        case 6: return launch(PsdSchurMma2Kernel<6>);
        case 7: return launch(PsdSchurMma2Kernel<7>);
        default: return launch(PsdSchurMma2Kernel<8>);
      }
    }
    switch (nt) {
      case 1: return launch(PsdSchurMmaKernel<1>);
      case 2: return launch(PsdSchurMmaKernel<2>);
      case 3: return launch(PsdSchurMmaKernel<3>);
      default: return launch(PsdSchurMmaKernel<4>);
    }
  }
  // LP / SOC cones: warp layout; the team version of the LMI Schur kernel keeps the CTA layout (its register tiles
  // and staging groups are sized for 128 threads)
  Geometry g = MakeGeometry(batch, SchurSmemBytes(c));
  if (c.type == CXB_CONE_PSD && g.warp) {
    g.warp = false;
    g.threads = kThreads;
    g.grid = batch;
    g.smem = SchurSmemBytes(c);
  }
  if (g.warp) {
    int rc = EnsureSmem(SchurKernel<true>, g.smem);
    if (rc) return rc;
    CountLaunch(); SchurKernel<true><<<g.grid, g.threads, g.smem, AsStream(stream)>>>(
        batch, g.per, c, dG, ldg, gstride, dAW, dAQc, vstride, d_scal, sstride, accumulate, d_active);
  } else {
    int rc = EnsureSmem(SchurKernel<false>, g.smem);
    if (rc) return rc;
    CountLaunch(); SchurKernel<false><<<g.grid, g.threads, g.smem, AsStream(stream)>>>(
        batch, g.per, c, dG, ldg, gstride, dAW, dAQc, vstride, d_scal, sstride, accumulate, d_active);
  }
  return LaunchStatus();
}

void cxb_set_small_psd_mma(int enabled) { g_small_psd_mma = enabled; }
void cxb_set_small_fused_launches(int enabled) { g_small_fused = enabled; }
void cxb_set_small_cone_threads(int threads) {
  if (threads == 32 || threads == 64 || threads == 128) g_spectral_threads = threads;
}
void cxb_set_small_team_mode(int mode) { g_small_team_mode = mode; }

int cxb_small_eigen(void* stream, int batch, const cxb_small_cone* cone, const double* dy, long ystride,
                    double c_weight, const double* d_cw, double* d_out4, long ostride,
                    const int* d_active) {
  if (batch <= 0) return 0;
  if (!ValidCone(cone)) return -1;
  const ConeArgs c = Convert(cone);
  const Geometry g = MakeGeometry(batch, SpectralSmemBytes(c), false, g_spectral_threads);
  if (g.warp) {
    int rc = EnsureSmem(EigenKernel<true>, g.smem);
    if (rc) return rc;
    CountLaunch(); EigenKernel<true><<<g.grid, g.threads, g.smem, AsStream(stream)>>>(
        batch, g.per, c, dy, ystride, c_weight, d_cw, d_out4, ostride, d_active);
  } else {
    int rc = EnsureSmem(EigenKernel<false>, g.smem);
    if (rc) return rc;
    CountLaunch(); EigenKernel<false><<<g.grid, g.threads, g.smem, AsStream(stream)>>>(
        batch, g.per, c, dy, ystride, c_weight, d_cw, d_out4, ostride, d_active);
  }
  return LaunchStatus();
}

int cxb_small_prepare(void* stream, int batch, const cxb_small_cone* cone, const double* dy, long ystride,
                      int affine, double c_weight, const double* d_cw, double e_weight, double* d_out2,
                      long ostride, const int* d_active) {
  if (batch <= 0) return 0;
  if (!ValidCone(cone)) return -1;
  const ConeArgs c = Convert(cone);
  const Geometry g = MakeGeometry(batch, SpectralSmemBytes(c), false, g_spectral_threads);
  if (g.warp) {
    int rc = EnsureSmem(PrepareKernel<true>, g.smem);
    if (rc) return rc;
    CountLaunch(); PrepareKernel<true><<<g.grid, g.threads, g.smem, AsStream(stream)>>>(
        batch, g.per, c, dy, ystride, affine, c_weight, d_cw, e_weight, d_out2, ostride, d_active);
  } else {
    int rc = EnsureSmem(PrepareKernel<false>, g.smem);
    if (rc) return rc;
    CountLaunch(); PrepareKernel<false><<<g.grid, g.threads, g.smem, AsStream(stream)>>>(
        batch, g.per, c, dy, ystride, affine, c_weight, d_cw, e_weight, d_out2, ostride, d_active);
  }
  return LaunchStatus();
}

int cxb_small_take_step(void* stream, int batch, const cxb_small_cone* cone, double step,
                        const double* d_step, double e_weight, int* d_info, const int* d_active) {
  if (batch <= 0) return 0;
  if (!ValidCone(cone)) return -1;
  if (cone->type == CXB_CONE_PSD && !d_info) return -1;
  const ConeArgs c = Convert(cone);
  const Geometry g = MakeGeometry(batch, SmemBytes(c));
  if (g.warp) {
    int rc = EnsureSmem(TakeStepKernel<true>, g.smem);
    if (rc) return rc;
    CountLaunch(); TakeStepKernel<true><<<g.grid, g.threads, g.smem, AsStream(stream)>>>(
        batch, g.per, c, step, d_step, e_weight, d_info, d_active);
  } else {
    int rc = EnsureSmem(TakeStepKernel<false>, g.smem);
    if (rc) return rc;
    CountLaunch(); TakeStepKernel<false><<<g.grid, g.threads, g.smem, AsStream(stream)>>>(
        batch, g.per, c, step, d_step, e_weight, d_info, d_active);
  }
  return LaunchStatus();
}

// ---- the same operations on a list of cones of every program, one launch per kMaxFused cones ----------------------
int cxb_small_set_identity_multi(void* stream, int batch, int ncones, const cxb_small_cone* cones,
                                 const int* d_active) {
  if (batch <= 0 || ncones <= 0) return 0;
  if (!cones) return -1;
  for (int first = 0; first < ncones; first += kMaxFused) {
    const int count = ncones - first < kMaxFused ? ncones - first : kMaxFused;
    if (!FusedLayout(batch)) {
      for (int k = 0; k < count; k++) {
        int rc = cxb_small_set_identity(stream, batch, cones + first + k, d_active);
        if (rc) return rc;
      }
      continue;
    }
    ConeList l;
    size_t smem;
    if (!MakeList(count, cones + first, [](const ConeArgs&) { return sizeof(double) * 64; }, &l, &smem)) return -1;
    CountLaunch();
    SetIdentityMultiKernel<<<dim3(batch, count), kThreads, smem, AsStream(stream)>>>(batch, (long)(smem / 8), l,
                                                                                     d_active);
    int rc = LaunchStatus();
    if (rc) return rc;
  }
  return 0;
}

int cxb_small_eigen_multi(void* stream, int batch, int ncones, const cxb_small_cone* cones, const double* dy,
                          long ystride, double c_weight, const double* d_cw, double* d_out4, long ostride,
                          const int* d_active) {
  if (batch <= 0 || ncones <= 0) return 0;
  if (!cones) return -1;
  for (int first = 0; first < ncones; first += kMaxFused) {
    const int count = ncones - first < kMaxFused ? ncones - first : kMaxFused;
    if (!FusedLayout(batch)) {
      for (int k = 0; k < count; k++) {
        int rc = cxb_small_eigen(stream, batch, cones + first + k, dy, ystride, c_weight, d_cw,
                                 d_out4 + 4 * (first + k), ostride, d_active);
        if (rc) return rc;
      }
      continue;
    }
    ConeList l;
    size_t smem;
    if (!MakeList(count, cones + first, SpectralSmemBytes, &l, &smem)) return -1;
    int rc = EnsureSmem(EigenMultiKernel, smem);
    if (rc) return rc;
    CountLaunch();
    EigenMultiKernel<<<dim3(batch, count), g_spectral_threads, smem, AsStream(stream)>>>(
        batch, (long)(smem / 8), l, dy, ystride, c_weight, d_cw, d_out4 + 4 * first, ostride, d_active);
    rc = LaunchStatus();
    if (rc) return rc;
  }
  return 0;
}

int cxb_small_prepare_multi(void* stream, int batch, int ncones, const cxb_small_cone* cones, const double* dy,
                            long ystride, int affine, double c_weight, const double* d_cw, double e_weight,
                            double* d_out2, long ostride, const int* d_active) {
  if (batch <= 0 || ncones <= 0) return 0;
  if (!cones) return -1;
  for (int first = 0; first < ncones; first += kMaxFused) {
    const int count = ncones - first < kMaxFused ? ncones - first : kMaxFused;
    if (!FusedLayout(batch)) {
      for (int k = 0; k < count; k++) {
        int rc = cxb_small_prepare(stream, batch, cones + first + k, dy, ystride, affine, c_weight, d_cw, e_weight,
                                   d_out2 + 4 * (first + k), ostride, d_active);
        if (rc) return rc;
      }
      continue;
    }
    ConeList l;
    size_t smem;
    if (!MakeList(count, cones + first, SpectralSmemBytes, &l, &smem)) return -1;
    int rc = EnsureSmem(PrepareMultiKernel, smem);
    if (rc) return rc;
    CountLaunch();
    PrepareMultiKernel<<<dim3(batch, count), g_spectral_threads, smem, AsStream(stream)>>>(
        batch, (long)(smem / 8), l, dy, ystride, affine, c_weight, d_cw, e_weight, d_out2 + 4 * first, ostride,
        d_active);
    rc = LaunchStatus();
    if (rc) return rc;
  }
  return 0;
}

int cxb_small_take_step_multi(void* stream, int batch, int ncones, const cxb_small_cone* cones, double step,
                              const double* d_step, double e_weight, int* d_info, const int* d_active) {
  if (batch <= 0 || ncones <= 0) return 0;
  if (!cones) return -1;
  for (int first = 0; first < ncones; first += kMaxFused) {
    const int count = ncones - first < kMaxFused ? ncones - first : kMaxFused;
    bool psd = false;
    for (int k = 0; k < count; k++) psd = psd || cones[first + k].type == CXB_CONE_PSD;
    if (psd && !d_info) return -1;
    if (!FusedLayout(batch)) {
      for (int k = 0; k < count; k++) {
        int rc = cxb_small_take_step(stream, batch, cones + first + k, step, d_step, e_weight, d_info, d_active);
        if (rc) return rc;
      }
      continue;
    }
    ConeList l;
    size_t smem;
    if (!MakeList(count, cones + first, SmemBytes, &l, &smem)) return -1;
    int rc = EnsureSmem(TakeStepMultiKernel, smem);
    if (rc) return rc;
    CountLaunch();
    TakeStepMultiKernel<<<dim3(batch, count), kThreads, smem, AsStream(stream)>>>(batch, (long)(smem / 8), l, step,
                                                                                  d_step, e_weight, d_info, d_active);
    rc = LaunchStatus();
    if (rc) return rc;
  }
  return 0;
}

int cxb_small_potrf_blocked(void* stream, int batch, int N, double* dH, long ldh, long hstride, int* d_info,
                            const int* d_active) {
  if (batch <= 0 || N <= 0) return 0;
  const size_t smem = sizeof(double) * BlockedKktSmemDoubles(N, false);
  int rc = EnsureSmem(BlockedPotrfKernel, smem);
  if (rc) return rc;
  CountLaunch();
  BlockedPotrfKernel<<<batch, kThreads, smem, AsStream(stream)>>>(N, dH, ldh, hstride, d_info, d_active);
  return LaunchStatus();
}

int cxb_small_potrf(void* stream, int batch, int N, double* dH, long ldh, long hstride, int* d_info,
                    const int* d_active) {
  if (batch <= 0 || N <= 0) return 0;
  const Geometry g = MakeGeometry(batch, sizeof(double) * (64 + (size_t)N * N));
  if (g.smem > kMaxSmemBytes) return cxb_small_potrf_blocked(stream, batch, N, dH, ldh, hstride, d_info, d_active);
  if (g.warp) {
    int rc = EnsureSmem(PotrfKernel<true>, g.smem);
    if (rc) return rc;
    CountLaunch(); PotrfKernel<true><<<g.grid, g.threads, g.smem, AsStream(stream)>>>(batch, g.per, N, dH, ldh, hstride,
                                                                                   d_info, d_active);
  } else {
    int rc = EnsureSmem(PotrfKernel<false>, g.smem);
    if (rc) return rc;
    CountLaunch(); PotrfKernel<false><<<g.grid, g.threads, g.smem, AsStream(stream)>>>(batch, g.per, N, dH, ldh, hstride,
                                                                                    d_info, d_active);
  }
  return LaunchStatus();
}

int cxb_small_potrs(void* stream, int batch, int N, const double* dL, long ldl, long lstride, double* dX,
                    long xstride, const int* d_active) {
  if (batch <= 0 || N <= 0) return 0;
  const Geometry g = MakeGeometry(batch, sizeof(double) * (64 + (size_t)N), /*chain_only=*/true);
  if (g.warp) {
    int rc = EnsureSmem(PotrsKernel<true>, g.smem);
    if (rc) return rc;
    CountLaunch(); PotrsKernel<true><<<g.grid, g.threads, g.smem, AsStream(stream)>>>(batch, g.per, N, dL, ldl, lstride, dX,
                                                                                   xstride, d_active);
  } else {
    int rc = EnsureSmem(PotrsKernel<false>, g.smem);
    if (rc) return rc;
    CountLaunch(); PotrsKernel<false><<<g.grid, g.threads, g.smem, AsStream(stream)>>>(batch, g.per, N, dL, ldl, lstride, dX,
                                                                                    xstride, d_active);
  }
  return LaunchStatus();
}

int cxb_small_ldlt_blocked(void* stream, int batch, int N, const double* dK, long ldk, long kstride, double* dL,
                           long ldl, long lstride, int* d_perm, long pstride, double* d_signs, long sstride,
                           int* d_info, const int* d_active) {
  if (batch <= 0 || N <= 0) return 0;
  const size_t smem = sizeof(double) * BlockedKktSmemDoubles(N, true);
  int rc = EnsureSmem(BlockedLdltKernel, smem);
  if (rc) return rc;
  CountLaunch();
  BlockedLdltKernel<<<batch, kThreads, smem, AsStream(stream)>>>(N, dK, ldk, kstride, dL, ldl, lstride, d_perm, pstride,
                                                                d_signs, sstride, d_info, d_active);
  return LaunchStatus();
}

int cxb_small_ldlt(void* stream, int batch, int N, const double* dK, long ldk, long kstride, double* dL, long ldl,
                   long lstride, int* d_perm, long pstride, double* d_signs, long sstride, int* d_info,
                   const int* d_active) {
  if (batch <= 0 || N <= 0) return 0;
  const Geometry g = MakeGeometry(batch, sizeof(double) * (64 + (size_t)LdltSmemDoubles(N)));
  if (g.smem > kMaxSmemBytes)
    return cxb_small_ldlt_blocked(stream, batch, N, dK, ldk, kstride, dL, ldl, lstride, d_perm, pstride, d_signs,
                                  sstride, d_info, d_active);
  if (g.warp) {
    int rc = EnsureSmem(LdltKernel<true>, g.smem);
    if (rc) return rc;
    CountLaunch(); LdltKernel<true><<<g.grid, g.threads, g.smem, AsStream(stream)>>>(
        batch, g.per, N, dK, ldk, kstride, dL, ldl, lstride, d_perm, pstride, d_signs, sstride, d_info, d_active);
  } else {
    int rc = EnsureSmem(LdltKernel<false>, g.smem);
    if (rc) return rc;
    CountLaunch(); LdltKernel<false><<<g.grid, g.threads, g.smem, AsStream(stream)>>>(
        batch, g.per, N, dK, ldk, kstride, dL, ldl, lstride, d_perm, pstride, d_signs, sstride, d_info, d_active);
  }
  return LaunchStatus();
}

int cxb_small_ldlt_solve(void* stream, int batch, int N, const double* dL, long ldl, long lstride, const int* d_perm,
                         long pstride, const double* d_signs, long sstride, double* dX, long xstride,
                         const int* d_active) {
  if (batch <= 0 || N <= 0) return 0;
  const Geometry g = MakeGeometry(batch, sizeof(double) * (64 + (size_t)N), /*chain_only=*/true);
  if (g.warp) {
    int rc = EnsureSmem(LdltSolveKernel<true>, g.smem);
    if (rc) return rc;
    CountLaunch(); LdltSolveKernel<true><<<g.grid, g.threads, g.smem, AsStream(stream)>>>(
        batch, g.per, N, dL, ldl, lstride, d_perm, pstride, d_signs, sstride, dX, xstride, d_active);
  } else {
    int rc = EnsureSmem(LdltSolveKernel<false>, g.smem);
    if (rc) return rc;
    CountLaunch(); LdltSolveKernel<false><<<g.grid, g.threads, g.smem, AsStream(stream)>>>(
        batch, g.per, N, dL, ldl, lstride, d_perm, pstride, d_signs, sstride, dX, xstride, d_active);
  }
  return LaunchStatus();
}

int cxb_small_gather(void* stream, int batch, int count, const int* d_idx, double* dy, long ystride, long dst,
                     const int* d_active) {
  if (batch <= 0 || count <= 0) return 0;
  if (!d_idx || !dy || dst < 0 || ystride < dst + count) return -1;
  CountLaunch();
  GatherKernel<<<batch, kThreads, 0, AsStream(stream)>>>(count, d_idx, dy, ystride, dst, d_active);
  return LaunchStatus();
}

int cxb_small_scatter_schur(void* stream, int batch, int ncones, const int* d_cones, const int* d_idx, const double* dS,
                            long sstride, int m, double* dH, long ldh, long hstride, double* dAW, double* dAQc,
                            long vstride, double* d_scal, long scal_stride, int accumulate, const int* d_active) {
  if (batch <= 0 || (ncones <= 0 && accumulate)) return 0;
  if (m < 1 || ldh < m || !dH || !dAW || !dAQc || !d_scal || (ncones > 0 && (!d_cones || !d_idx || !dS))) return -1;
  CountLaunch();
  ScatterSchurKernel<<<batch, kThreads, 0, AsStream(stream)>>>(ncones, d_cones, d_idx, dS, sstride, m, dH, ldh, hstride,
                                                               dAW, dAQc, vstride, d_scal, scal_stride, accumulate,
                                                               d_active);
  return LaunchStatus();
}

int cxb_batched_lincomb(void* stream, int batch, int n, const double* d_a, const double* dx, long xs,
                        const double* d_b, const double* dy, long ys, const double* d_c, const double* dz,
                        long zs, double* d_out, long os, const int* d_active) {
  if (batch <= 0 || n <= 0) return 0;
  dim3 grid((n + 127) / 128, batch);
  CountLaunch(); LincombKernel<<<grid, 128, 0, AsStream(stream)>>>(n, d_a, dx, xs, d_b, dy, ys, d_c, dz, zs, d_out, os,
                                                     d_active);
  return LaunchStatus();
}

int cxb_batched_dot(void* stream, int batch, int n, const double* dx, long xs, const double* dy, long ys,
                    double* d_out, long ostride) {
  if (batch <= 0) return 0;
  CountLaunch(); BatchedDotKernel<<<batch, kThreads, 0, AsStream(stream)>>>(n, dx, xs, dy, ys, d_out, ostride);
  return LaunchStatus();
}

}  // extern "C"

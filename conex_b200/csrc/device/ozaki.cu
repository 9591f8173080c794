// K2 of the symmetric Schur assembly on the 8-bit integer tensor cores: the lower triangle of the Gram matrix
// H = X^T X of an FP64 operand X (K x M, column-major), computed by FP64 emulation (the Ozaki scheme).
//
// Slicing. Column j of X is scaled by its own power of two, 2^-e_j with max_k |X[k, j]| < 2^e_j, and cut into
// kSlices signed 7-bit digits by round-to-nearest:
//   r_0 = X[k, j] 2^(6 - e_j),  D_t = rint(r_{t-1}),  r_t = 128 (r_{t-1} - D_t)        (t = 1 .. s)
// so X[k, j] = 2^(e_j - 6) (sum_t D_t 2^(-7 (t - 1)) + r_s 2^(-7 s)) with every D_t and r_t in [-64, 64]. Every step
// is exact in FP64 (r - rint(r) is representable, the scaling is by powers of two), so the digits are a pure function
// of X: the same on every device, rank and run.
//
// Products. X[k, i] X[k, j] = 2^(e_i + e_j - 12) sum_{t,u} D_t D_u 2^(-7 (t + u - 2)). Pairs of one level
// l = t + u - 2 share the scale 2^(-7 l); the levels l = 0 .. s - 1 are kept (s (s + 1) / 2 = 36 slice products for
// s = 8), each in its own int32 accumulator. A level holds at most s pairs of products |D_t D_u| <= 2^12, so a K
// range of 2^15 sums to at most 8 * 2^12 * 2^15 = 2^30 < 2^31: K is cut into chunks of kChunk = 2^15 and the level
// sums of each chunk are converted to FP64 and added, chunk after chunk and level after level in a fixed order, so
// the result is bit-identical from run to run.
//
// Error bound (per entry, exact arithmetic on the digits, u = 2^-53). The terms not computed are the pairs of levels
// s .. 2s - 2 (at most s - 1 pairs of at most 2^12 per level, geometric in 2^-7) and the two cross terms with the
// remainders r_s (each at most 64 * 64.01 * 2^-7s); per k they sum to at most 9.1 * 2^12 * 2^(-7 s) * 2^(e_i + e_j - 12),
// and with 2^e <= 2 max|X[:, j]|:
//   |H_ij - H~_ij| <= K * 36.4 * 2^(-7 s) * max|X[:, i]| max|X[:, j]| = K * 2^(-50.8) * max|X[:, i]| max|X[:, j]|  (s = 8)
// plus the FP64 rounding of the final sums (one rounding per level and chunk, K / 2^15 * s additions). The FP64 DMMA
// product's own worst-case bound is gamma_K sum_k |X[k, i] X[k, j]| ~ K u sum_k |X[k, i]| |X[k, j]|: the emulated
// result is within 4.6 K u max|X_i| max|X_j| <= 4.6 K u ||X_i|| ||X_j||, the norm-wise form of the FP64 bound up to a
// factor 4.6. Each further slice would cost s + 1 more slice products for another factor 2^-7; s = 8 also uses the
// tensor memory exactly (8 levels x 64 columns = 512 columns).
//
// Kernel. One CTA per 128 x 64 output tile of the lower triangle (rows i, columns j), one CTA per SM:
//   warp 0: bulk copies (TMA) of one 32-byte k-step of all 8 slices of the 128 A rows and the 64 B rows (48 KB per
//           stage, 4 stages) into an mbarrier ring;
//   warp 1: allocates the 512 TMEM columns and issues the 36 tcgen05.mma.kind::i8 (M 128, N 64, K 32) of each k-step
//           into the 8 level accumulators; tcgen05.commit frees a stage when its MMAs are done and, at the end of a
//           chunk, hands the accumulators to the epilogue;
//   warps 2-5: tcgen05.ld the level sums of each chunk (one TMEM lane = one output row per thread), convert and add
//           them into FP64 registers, release the accumulators, and finally scale by 2^(e_i + e_j - 12) and store.
//
// Slice layout. The slicing pass writes the digits in the order the MMAs read them from shared memory, so that every
// stage is a few large contiguous copies: rows in blocks of 128 (zero-padded), and for each row block and k-step the
// 8 slices one after the other, each 128 rows x 32 bytes in the 32-byte swizzle of the MMA's K-major operand (16-byte
// half h of row r at h ^ ((r >> 2) & 1)). A stage is then one 32 KB copy for the A rows and eight 2 KB copies for the
// B rows. (A 3-D tensor-map box over a plain [slice][row][k] layout reads 32-byte pieces of rows 2 MB apart, 1536 of
// them per stage: 0.64 POP/s and twice the DMMA Gram's time at C2, measured on a B200, 1000 W, 1965 MHz.)
#include "common.cuh"
#include "device_api.h"

namespace cxb {
namespace {

constexpr int kSlices = 8;          // s
constexpr int kLevels = kSlices;    // levels l = 0 .. s - 1
constexpr int kTileM = 128, kTileN = 64, kStepK = 32;
constexpr int kStages = 4;
constexpr int kChunkSteps = (1 << 15) / kStepK;
constexpr int kStageABytes = kSlices * kTileM * kStepK;   // 32 KB
constexpr int kStageBBytes = kSlices * kTileN * kStepK;   // 16 KB
constexpr int kStageBytes = kStageABytes + kStageBBytes;
constexpr int kThreads = 192;
constexpr size_t kSmemBytes = (size_t)kStages * kStageBytes + 256 + 1024;  // stages + barriers + alignment slack
static_assert(kLevels * kTileN <= 512, "level accumulators exceed the tensor memory");

__device__ __forceinline__ uint32_t Smem(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void BarInit(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(Smem(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void BarExpectTx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(Smem(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void BarArrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(Smem(bar)) : "memory");
}
__device__ __forceinline__ void BarWait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "OZ_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra OZ_DONE;\n\t"
      "bra OZ_WAIT;\n\t"
      "OZ_DONE:\n\t"
      "}" ::"r"(Smem(bar)),
      "r"(parity)
      : "memory");
}

__device__ __forceinline__ void BulkLoad(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(Smem(dst)), "l"(src), "r"(bytes), "r"(Smem(bar))
               : "memory");
}

// Shared-memory matrix descriptor: K-major operand, 32-byte swizzle (8-row atoms of 32 bytes, atoms 256 bytes apart)
__device__ __forceinline__ uint64_t SmemDescSw32(uint32_t addr) {
  uint64_t d = 0;
  d |= (uint64_t)((addr >> 4) & 0x3FFF);       // start address
  d |= (uint64_t)1 << 16;                      // leading byte offset (unused: K of one MMA is one swizzle row)
  d |= (uint64_t)(256 >> 4) << 32;             // stride byte offset: next 8 rows
  d |= (uint64_t)1 << 46;                      // descriptor version (sm_100)
  d |= (uint64_t)6 << 61;                      // swizzle: 32 B
  return d;
}

// Instruction descriptor of tcgen05.mma.kind::i8: s32 accumulator, signed 8-bit A and B, both K-major, M x N
constexpr uint32_t kInstrDesc = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kTileN >> 3) << 17) |
                                ((uint32_t)(kTileM >> 4) << 24);

__device__ __forceinline__ void MmaI8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(kInstrDesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void MmaCommit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(Smem(bar))
               : "memory");
}
__device__ __forceinline__ void FenceBefore() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void FenceAfter() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// 32 consecutive TMEM columns of this warp's 32 lanes
__device__ __forceinline__ void TmemLoad32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// e_j with max_k |X[k, j]| < 2^e_j (0 for an all-zero column); one block per column
__global__ void __launch_bounds__(256) ColumnExponentKernel(long K, const double* __restrict__ X, long ldx, int* exps) {
  const double* x = X + (long)blockIdx.x * ldx;
  double mx = 0.0;
  for (long k = threadIdx.x; k < K; k += 256) mx = fmax(mx, fabs(x[k]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  __shared__ double part[8];
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = mx;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; w++) mx = fmax(mx, part[w]);
    int e = 0;
    if (mx > 0.0) frexp(mx, &e);
    exps[blockIdx.x] = e;
  }
}

// Digits of rows j = 128 blockIdx.y + threadIdx.x, k-step blockIdx.x (32 k), in the layout described above
__global__ void __launch_bounds__(128) SliceKernel(long K, const double* __restrict__ X, long ldx,
                                                   const int* __restrict__ exps, int M, long ksteps, int8_t* slices) {
  const int r = threadIdx.x;
  const int j = blockIdx.y * kTileM + r;
  const long ks = blockIdx.x;
  uint32_t words[kSlices][8];
#pragma unroll
  for (int t = 0; t < kSlices; t++)
#pragma unroll
    for (int w = 0; w < 8; w++) words[t][w] = 0;
  if (j < M) {
    // x 2^(6 - e) as (x s1) s2 with powers of two s1, s2: the first product is exact, the second rounds once, so this is
    // ldexp(x, 6 - e) (2^(6 - e) itself exceeds the double range only for columns below 2^-1017)
    const int p = 6 - exps[j];
    const int p1 = p > 1023 ? 1000 : 0;
    const double s1 = __longlong_as_double((long long)(1023 + p1) << 52);
    const double s2 = __longlong_as_double((long long)(1023 + p - p1) << 52);
    const double* x = X + (long)j * ldx + ks * kStepK;
    const int valid = (int)min((long)kStepK, K - ks * kStepK);
#pragma unroll
    for (int q = 0; q < kStepK; q++) {
      double r0 = q < valid ? (x[q] * s1) * s2 : 0.0;
#pragma unroll
      for (int t = 0; t < kSlices; t++) {
        const double d = rint(r0);
        r0 = (r0 - d) * 128.0;
        words[t][q >> 2] |= ((uint32_t)(int)d & 0xFFu) << (8 * (q & 3));
      }
    }
  }
  const int sw = (r >> 2) & 1;
  int8_t* base = slices + ((long)blockIdx.y * ksteps + ks) * kSlices * (kTileM * kStepK) + r * kStepK;
#pragma unroll
  for (int t = 0; t < kSlices; t++) {
    uint4* row = reinterpret_cast<uint4*>(base + t * (kTileM * kStepK));
    row[sw] = make_uint4(words[t][0], words[t][1], words[t][2], words[t][3]);
    row[sw ^ 1] = make_uint4(words[t][4], words[t][5], words[t][6], words[t][7]);
  }
}

struct GramArgs {
  int M, N, tiles_m;
  int ksteps;
  const int8_t* slices;
  const int* exps;
  double* H;
  long ldh;
};

__global__ void __launch_bounds__(kThreads, 1)
    GramI8Kernel(const GramArgs g) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + kStages * kStageBytes);
  uint64_t* empty = full + kStages;
  uint64_t* acc_full = empty + kStages;
  uint64_t* acc_empty = acc_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 1);

  // blockIdx.x enumerates the lower tiles column by column: tile column tn holds rows tm >= (tn * 64) / 128
  int tn = 0, rem = blockIdx.x;
  for (;;) {
    const int count = g.tiles_m - (tn * kTileN) / kTileM;
    if (rem < count) break;
    rem -= count;
    tn++;
  }
  const int tm = (tn * kTileN) / kTileM + rem;
  const int m0 = tm * kTileM, n0 = tn * kTileN;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; s++) {
      BarInit(full + s, 1);
      BarInit(empty + s, 1);
    }
    BarInit(acc_full, 1);
    BarInit(acc_empty, 128);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(Smem(tmem_slot))
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  FenceBefore();
  __syncthreads();
  FenceAfter();
  const uint32_t tmem = *tmem_slot;
  const int nchunks = (g.ksteps + kChunkSteps - 1) / kChunkSteps;

  if (warp == 0) {
    if (lane == 0) {
      // A: row block tm whole; B: the 64-row half (n0 % 128) / 64 of row block n0 / 128, slice by slice
      const int8_t* a_src = g.slices + (long)tm * g.ksteps * kStageABytes;
      const int8_t* b_src = g.slices + (long)(n0 / kTileM) * g.ksteps * kStageABytes + (n0 % kTileM) * kStepK;
      for (int ks = 0; ks < g.ksteps; ks++) {
        const int s = ks % kStages;
        if (ks >= kStages) BarWait(empty + s, (uint32_t)(((ks / kStages) + 1) & 1));
        uint8_t* st = smem + s * kStageBytes;
        BarExpectTx(full + s, kStageBytes);
        BulkLoad(st, a_src + (long)ks * kStageABytes, kStageABytes, full + s);
#pragma unroll
        for (int t = 0; t < kSlices; t++) {
          BulkLoad(st + kStageABytes + t * (kTileN * kStepK), b_src + (long)ks * kStageABytes + t * (kTileM * kStepK),
                   kTileN * kStepK, full + s);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      for (int c = 0; c < nchunks; c++) {
        if (c > 0) {
          BarWait(acc_empty, (uint32_t)((c - 1) & 1));
          FenceAfter();
        }
        const int ks_end = min(g.ksteps, (c + 1) * kChunkSteps);
        for (int ks = c * kChunkSteps; ks < ks_end; ks++) {
          const int s = ks % kStages;
          BarWait(full + s, (uint32_t)((ks / kStages) & 1));
          FenceAfter();
          const uint32_t a_base = Smem(smem + s * kStageBytes);
          const uint32_t b_base = a_base + kStageABytes;
          const uint32_t first = (ks == c * kChunkSteps) ? 1u : 0u;
#pragma unroll
          for (int l = 0; l < kLevels; l++) {
#pragma unroll
            for (int t = 0; t <= l; t++) {
              const int u = l - t;
              MmaI8(tmem + l * kTileN, SmemDescSw32(a_base + t * (kTileM * kStepK)),
                    SmemDescSw32(b_base + u * (kTileN * kStepK)), (first && t == 0) ? 0u : 1u);
            }
          }
          MmaCommit(empty + s);
        }
        MmaCommit(acc_full);
      }
    }
  } else {
    // epilogue: TMEM lane quarter (warp % 4) = output rows 32 (warp % 4) .. + 31
    const int quarter = warp & 3;
    const uint32_t lane_base = tmem + ((uint32_t)(quarter * 32) << 16);
    double acc[kTileN];
#pragma unroll
    for (int c = 0; c < kTileN; c++) acc[c] = 0.0;
    for (int c = 0; c < nchunks; c++) {
      BarWait(acc_full, (uint32_t)(c & 1));
      FenceAfter();
      double scale = 1.0;
#pragma unroll 1
      for (int l = 0; l < kLevels; l++) {
#pragma unroll
        for (int h = 0; h < 2; h++) {
          uint32_t v[32];
          TmemLoad32(lane_base + l * kTileN + h * 32, v);
#pragma unroll
          for (int q = 0; q < 32; q++) acc[h * 32 + q] += scale * (double)(int)v[q];
        }
        scale *= 0.0078125;  // 2^-7
      }
      FenceBefore();
      BarArrive(acc_empty);
    }
    const int r = m0 + quarter * 32 + lane;
    if (r < g.M) {
      const int er = g.exps[r] - 12;
#pragma unroll
      for (int q = 0; q < kTileN; q++) {
        const int col = n0 + q;
        if (col < g.N && col <= r) g.H[(long)col * g.ldh + r] = ldexp(acc[q], er + g.exps[col]);
      }
    }
  }
  FenceBefore();
  __syncthreads();
  if (warp == 1) {
    FenceAfter();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
  }
}

long KSteps(long K) { return (K + kStepK - 1) / kStepK; }
size_t SliceBytes(int M, long K) { return (size_t)((M + kTileM - 1) / kTileM) * KSteps(K) * kStageABytes; }

}  // namespace

size_t GramEmulatedWorkspace(int M, long K) { return SliceBytes(M, K) + sizeof(int) * (size_t)M; }

int GramSlices(cudaStream_t s, int M, long K, const double* X, long ldx, void* work) {
  if (M < 1 || K < 16 || (K % 16) != 0 || ldx < K || KSteps(K) > (1L << 30)) return -1;
  int8_t* slices = static_cast<int8_t*>(work);
  int* exps = reinterpret_cast<int*>(slices + SliceBytes(M, K));
  CountLaunch(); ColumnExponentKernel<<<M, 256, 0, s>>>(K, X, ldx, exps);
  const int row_blocks = (M + kTileM - 1) / kTileM;
  CountLaunch(); SliceKernel<<<dim3((unsigned)KSteps(K), row_blocks), kTileM, 0, s>>>(K, X, ldx, exps, M, KSteps(K),
                                                                                        slices);
  return LaunchStatus();
}

int GramEmulated(cudaStream_t s, int M, int N, long K, const double* X, long ldx, double* H, long ldh, void* work) {
  if (N < 1 || N > M || ldh < M) return -1;
  int rc = GramSlices(s, M, K, X, ldx, work);
  if (rc) return rc;
  static std::atomic<unsigned long long> configured{0};
  if (FirstUseOnCurrentDevice(configured)) {
    cudaFuncSetAttribute(GramI8Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes);
  }
  GramArgs g;
  g.M = M;
  g.N = N;
  g.tiles_m = (M + kTileM - 1) / kTileM;
  g.ksteps = (int)KSteps(K);
  g.slices = static_cast<const int8_t*>(work);
  g.exps = reinterpret_cast<const int*>(g.slices + SliceBytes(M, K));
  g.H = H;
  g.ldh = ldh;
  const int tiles_n = (N + kTileN - 1) / kTileN;
  long tiles = 0;
  for (int tn = 0; tn < tiles_n; tn++) tiles += g.tiles_m - (tn * kTileN) / kTileM;
  CountLaunch(); GramI8Kernel<<<(unsigned)tiles, kThreads, kSmemBytes, s>>>(g);
  return LaunchStatus();
}

}  // namespace cxb

extern "C" size_t cxb_gram_emulated_workspace(int M, long K) { return cxb::GramEmulatedWorkspace(M, K); }

extern "C" int cxb_gram_slices(void* stream, int M, long K, const double* dX, long ldx, void* dWork) {
  return cxb::GramSlices(cxb::AsStream(stream), M, K, dX, ldx, dWork);
}

extern "C" int cxb_gram_emulated(void* stream, int M, int N, long K, const double* dX, long ldx, double* dH, long ldh,
                                 void* dWork) {
  return cxb::GramEmulated(cxb::AsStream(stream), M, N, K, dX, ldx, dH, ldh, dWork);
}

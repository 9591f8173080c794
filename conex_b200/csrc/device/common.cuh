// Shared device helpers for the conex-b200 kernels (sm_100a only).
#pragma once
#include <atomic>
#include <cuda_runtime.h>
#include <stdint.h>

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "conex-b200 kernels are written for sm_100a (Blackwell B200) only"
#endif

namespace cxb {

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs

inline int LaunchStatus() {
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : static_cast<int>(e);
}

inline cudaStream_t AsStream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// Every kernel launch of the library is counted (reported by CONEXB200_LaunchCount / bench.py).
extern std::atomic<long> g_launch_count;
inline void CountLaunch() { g_launch_count.fetch_add(1, std::memory_order_relaxed); }

// Per-kernel attributes (cudaFuncSetAttribute) are per device: `mask` has one bit per device ordinal.
// Returns true the first time the calling thread's current device is seen (programs may be driven from
// several host threads and on several devices of one process, like the reference's Program objects).
inline bool FirstUseOnCurrentDevice(std::atomic<unsigned long long>& mask) {
  int device = 0;
  if (cudaGetDevice(&device) != cudaSuccess || device < 0 || device >= 64) return true;
  const unsigned long long bit = 1ull << device;
  if (mask.load(std::memory_order_acquire) & bit) return false;
  mask.fetch_or(bit, std::memory_order_acq_rel);
  return true;
}

// A high-priority side stream and two events for a look-ahead schedule: the next panel is factored on
// the side stream while the main stream applies the current one to the rest of the matrix. Meant to be
// held per host thread (a Program is single-threaded; programs driven from different threads get their
// own). Prepare() creates them on first use and re-creates them when the thread's current device changes.
struct LookAhead {
  cudaStream_t side = nullptr;
  cudaEvent_t updated = nullptr, factored = nullptr;
  int device = -1;
  bool Prepare() {
    int current = 0;
    if (cudaGetDevice(&current) != cudaSuccess) return false;
    if (side && device == current) return true;
    if (side) {  // the thread moved to another device: streams and events belong to the old one
      cudaStreamDestroy(side);
      cudaEventDestroy(updated);
      cudaEventDestroy(factored);
      side = nullptr;
    }
    device = current;
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);
    if (cudaStreamCreateWithPriority(&side, cudaStreamNonBlocking, hi) != cudaSuccess) return false;
    return cudaEventCreateWithFlags(&updated, cudaEventDisableTiming) == cudaSuccess &&
           cudaEventCreateWithFlags(&factored, cudaEventDisableTiming) == cudaSuccess;
  }
};

// ---- cp.async (LDGSTS) -------------------------------------------------------------------
// 16-byte copy with zero fill of the bytes beyond src_bytes (0, 8 or 16).
__device__ __forceinline__ void CpAsync16(void* smem, const void* gmem, int src_bytes) {
  const uint32_t s = static_cast<uint32_t>(__cvta_generic_to_shared(smem));
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(src_bytes));
}
// 8-byte copy with zero fill when src_bytes == 0.
__device__ __forceinline__ void CpAsync8(void* smem, const void* gmem, int src_bytes) {
  const uint32_t s = static_cast<uint32_t>(__cvta_generic_to_shared(smem));
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(s), "l"(gmem), "r"(src_bytes));
}
__device__ __forceinline__ void CpAsyncCommit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void CpAsyncWait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}

// ---- FP64 tensor core: D(8x8) += A(8x4) * B(4x8); SASS: DMMA.8x8x4 --------------------------
// lane l holds A[l/4][l%4], B[l%4][l/4], C[l/4][2*(l%4) + {0,1}].
__device__ __forceinline__ void Dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

// ---- reductions ------------------------------------------------------------------------------
__device__ __forceinline__ double WarpSum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Sum over the whole block; result valid in every thread. `scratch` holds >= 33 doubles.
__device__ __forceinline__ double BlockSum(double v, double* scratch) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nwarps = (blockDim.x + 31) >> 5;
  v = WarpSum(v);
  __syncthreads();
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  if (warp == 0) {
    double t = (lane < nwarps) ? scratch[lane] : 0.0;
    t = WarpSum(t);
    if (lane == 0) scratch[32] = t;
  }
  __syncthreads();
  return scratch[32];
}

}  // namespace cxb

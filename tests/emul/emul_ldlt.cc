// TEST INFRASTRUCTURE ONLY — never linked into libconex_b200.so.
//
// The batched regularised LDL^T of small KKT systems (SmallLdlt / SmallLdltSolve of
// conex_b200/csrc/device/small_cone_math.cuh) executed serially on the CPU, behind the same argument
// lists as cxb_small_ldlt / cxb_small_ldlt_solve (without the stream). Same serial stand-in for the
// team as tests/emul/emul_small.cc: every parallel loop runs in index order, every barrier is a no-op.
#include <cstddef>
#include <vector>

#include "../../conex_b200/csrc/device/small_cone_math.cuh"

namespace {

struct HostTeam {
  int size() const { return 128; }
  template <class F>
  void par(int n, F f) {
    for (int i = 0; i < n; i++) f(i);
  }
  template <class R, class F>
  void par2(int rows, int cols, R row_value, F f) {
    for (int i = 0; i < rows; i++) {
      const double rv = row_value(i);
      for (int c = 0; c < cols; c++) f(i, c, rv);
    }
  }
  template <class F>
  double sum(int n, F f) {
    double v = 0;
    for (int i = 0; i < n; i++) v += f(i);
    return v;
  }
  // index of the FIRST largest f(i), as the device teams
  template <class F>
  int argmax_first(int n, F f, double* vmax) {
    int best = 0;
    double bv = f(0);
    for (int i = 1; i < n; i++)
      if (f(i) > bv) {
        bv = f(i);
        best = i;
      }
    *vmax = bv;
    return best;
  }
  template <class F>
  void single(F f) {
    f();
  }
  template <class F>
  void warp0(F f) {
    f(*this);
  }
};

}  // namespace

using namespace cxb::small;

extern "C" {

int emul_small_ldlt(int batch, int N, const double* K, long ldk, long kstride, double* L, long ldl, long lstride,
                    int* perm, long pstride, double* signs, long sstride, int* info, const int* active) {
  HostTeam t;
  std::vector<double> sm((size_t)N * N + N);
  std::vector<int> at(N);
  for (int p = 0; p < batch; p++) {
    if (active && !active[p]) continue;
    info[p] = SmallLdlt(t, N, K + p * kstride, ldk, L + p * lstride, ldl, perm + p * pstride, signs + p * sstride,
                        sm.data(), sm.data() + (size_t)N * N, at.data());
  }
  return 0;
}

int emul_small_ldlt_solve(int batch, int N, const double* L, long ldl, long lstride, const int* perm, long pstride,
                          const double* signs, long sstride, double* X, long xstride, const int* active) {
  HostTeam t;
  std::vector<double> sm(N);
  for (int p = 0; p < batch; p++) {
    if (active && !active[p]) continue;
    SmallLdltSolve(t, N, L + p * lstride, ldl, perm + p * pstride, signs + p * sstride, X + p * xstride, sm.data());
  }
  return 0;
}

}  // extern "C"

// TEST INFRASTRUCTURE ONLY — never linked into libconex_b200.so.
//
// The blocked factorisations of KKT systems larger than shared memory (BlockedPotrf / BlockedLdlt of
// conex_b200/csrc/device/small_cone_math.cuh, with the plain-loop trailing update KktTrailingUpdateLoop in place of
// the DMMA tiles) executed serially on the CPU, behind the same argument lists as cxb_small_potrf_blocked /
// cxb_small_ldlt_blocked (without the stream). Same serial stand-in for the team as tests/emul/emul_ldlt.cc.
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

int emul_small_potrf_blocked(int batch, int N, double* H, long ldh, long hstride, int* info, const int* active) {
  HostTeam t;
  std::vector<double> sm(BlockedKktSmemDoubles());
  for (int p = 0; p < batch; p++) {
    if (active && !active[p]) continue;
    info[p] = BlockedPotrf(t, N, H + p * hstride, ldh, sm.data(), KktTrailingUpdateLoop());
  }
  return 0;
}

int emul_small_ldlt_blocked(int batch, int N, const double* K, long ldk, long kstride, double* L, long ldl,
                            long lstride, int* perm, long pstride, double* signs, long sstride, int* info,
                            const int* active) {
  HostTeam t;
  std::vector<double> sm(BlockedKktSmemDoubles()), sd(N);
  std::vector<int> at(N);
  for (int p = 0; p < batch; p++) {
    if (active && !active[p]) continue;
    info[p] = BlockedLdlt(t, N, K + p * kstride, ldk, L + p * lstride, ldl, perm + p * pstride, signs + p * sstride,
                          sm.data(), sd.data(), at.data(), KktTrailingUpdateLoop());
  }
  return 0;
}

}  // extern "C"

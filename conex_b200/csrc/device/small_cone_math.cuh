// Per-problem arithmetic of the small cones — LP cone, second-order cone, small dense PSD/LMI
// block — and of the small dense KKT system, written once against a "team" (team.cuh): every
// function below is executed by ONE CTA on ONE cone of ONE program; the kernels in small_cones.cu
// map blockIdx.x to the program of a batch. Used by
//   * the batched solver (many small multi-cone programs in lock step, BASELINE config 3), and
//   * the single-program LP / SOC plugins (batch of one).
//
// Reference arithmetic restated here (column-major FP64 throughout):
//   LP   conex/linear_constraint.cc:105-205        SOC  conex/soc_constraint.cc:115-262
//   PSD  conex/psd_constraint.cc:13-128, conex/dense_lmi_constraint.cc:8-103,
//        conex/exponential_map_pade.cc:10-32, conex/approximate_eigenvalues.cc:173-256
//   KKT  conex/block_triangular_operations.cc:114-219 (one dense supernode)
//
// Data layout of a cone with `rows` slack entries per variable (LP: n, SOC: n + 1, PSD: n * n):
//   data  = rows x (m + 1) column-major, columns 0..m-1 the operator, column m the affine term.
#pragma once
#include <math.h>

#ifdef __CUDACC__
#define CXB_HD __device__ __forceinline__
#define CXB_HOST_DEVICE __host__ __device__ inline
#else
#define CXB_HD inline
#define CXB_HOST_DEVICE inline
#endif

namespace cxb {
namespace small {

CXB_HD void Accumulate(double* dst, double v, bool acc) { *dst = acc ? *dst + v : v; }

// e -> (e % d, e / d) for 0 <= e < 2^31 with e / d < 2^22 (every use below: the quotient is a row or column index)
// without the ~25-instruction integer division by a run-time divisor — the element loops map a flat index to
// (row, column) for every element, and in the issue-bound kernels those two divisions were most of the instructions.
// The float product is off by less than one from the true quotient and one comparison each way makes it exact, so
// the loops visit the same elements in the same order.
struct Divider {
  int d;
  float inv;
  CXB_HD explicit Divider(int divisor) : d(divisor), inv(1.0f / (float)divisor) {}
  CXB_HD int quot(int e) const {
    int q = (int)(((float)e + 0.5f) * inv);
    const int r = e - q * d;
    if (r < 0) q--;
    if (r >= d) q++;
    return q;
  }
  CXB_HD int rem(int e) const { return e - quot(e) * d; }
};

// out[r] = sum_j data[r + j * rows] y[j] - k * data[r + m * rows]
template <class T>
CXB_HD void NegativeSlack(T& t, int rows, int m, const double* data, const double* y, double k,
                          double* out) {
  // Independent loads in flight per thread: the columns are 8 * rows bytes apart in HBM, and a loop that consumes each
  // load before issuing the next one pays the full memory latency m times per row (this phase reads the whole cone
  // data and was latency-bound: 1.6 TB/s with 32 warps per SM). Even row counts on 16-byte aligned data: two rows per
  // thread, eight 16-byte loads in flight. Same summation order per row.
#ifdef __CUDA_ARCH__
  if ((rows & 1) == 0 && (reinterpret_cast<unsigned long long>(data) & 15) == 0) {
    t.par(rows / 2, [&](int q) {
      const double2* col = reinterpret_cast<const double2*>(data) + q;
      const long stride = rows / 2;
      double s0 = 0, s1 = 0;
      int j = 0;
      for (; j + 8 <= m; j += 8) {
        double2 a[8];
#pragma unroll
        for (int u = 0; u < 8; u++) a[u] = col[(long)(j + u) * stride];
#pragma unroll
        for (int u = 0; u < 8; u++) {
          s0 += a[u].x * y[j + u];
          s1 += a[u].y * y[j + u];
        }
      }
      const double2 c = col[(long)m * stride];
      for (; j < m; j++) {
        const double2 a = col[(long)j * stride];
        s0 += a.x * y[j];
        s1 += a.y * y[j];
      }
      out[2 * q] = s0 - k * c.x;
      out[2 * q + 1] = s1 - k * c.y;
    });
    return;
  }
#endif
  t.par(rows, [&](int r) {
    double s = 0;
    int j = 0;
    for (; j + 8 <= m; j += 8) {
      double a[8];
#pragma unroll
      for (int u = 0; u < 8; u++) a[u] = data[(long)(j + u) * rows + r];
#pragma unroll
      for (int u = 0; u < 8; u++) s += a[u] * y[j + u];
    }
    const double c = data[(long)m * rows + r];
    for (; j < m; j++) s += data[(long)j * rows + r] * y[j];
    out[r] = s - k * c;
  });
}

// =================================================================================================
// LP cone. state: W[n], t1[n], t2[n].
// =================================================================================================
// sm: nullptr, or LpSchurSmemDoubles(n, m) doubles of team-shared scratch: the scaled operator [W A | W c] is staged
// there once (coalesced read of the cone data) and the m (m + 1) / 2 inner products run out of it; without it every
// pair re-reads two columns of the operator from global memory with a stride of n doubles between threads. Same
// products, same summation order.
CXB_HOST_DEVICE long LpSchurSmemDoubles(int n, int m) { return (long)(n | 1) * (m + 1); }
template <class T>
CXB_HD void LpSchur(T& t, int n, int m, const double* Ac, const double* W, double* G, long ldg,
                    double* AW, double* AQc, double* scal, bool acc, double* sm = nullptr) {
  if (sm != nullptr) {
    const int P = n | 1;  // odd pitch: threads on consecutive columns hit different banks
    const Divider by_n(n), by_m(m);
    t.par(n * (m + 1), [&](int e) {
      const int j = by_n.quot(e), r = e - j * n;
      sm[(long)j * P + r] = W[r] * Ac[e];
    });
    const double* wc = sm + (long)m * P;
    t.par(m * m, [&](int e) {
      const int j = by_m.quot(e), i = e - j * m;
      if (i < j) return;
      const double* ai = sm + (long)i * P;
      const double* aj = sm + (long)j * P;
      double s = 0;
      for (int r = 0; r < n; r++) s += ai[r] * aj[r];
      Accumulate(G + (long)j * ldg + i, s, acc);
    });
    t.par(m, [&](int j) {
      const double* aj = sm + (long)j * P;
      double aw = 0, aq = 0;
      for (int r = 0; r < n; r++) {
        aw += aj[r];
        aq += aj[r] * wc[r];
      }
      Accumulate(AW + j, aw, acc);
      Accumulate(AQc + j, aq, acc);
    });
    const double s1 = t.sum(n, [&](int r) { return wc[r]; });
    const double s2 = t.sum(n, [&](int r) { return wc[r] * wc[r]; });
    t.single([&]() {
      Accumulate(scal + 0, s1, acc);
      Accumulate(scal + 1, s2, acc);
    });
    return;
  }
  const double* c = Ac + (long)m * n;
  const Divider by_m(m);
  t.par(m * m, [&](int e) {
    const int j = by_m.quot(e), i = e - j * m;
    if (i < j) return;
    const double* ai = Ac + (long)i * n;
    const double* aj = Ac + (long)j * n;
    double s = 0;
    for (int r = 0; r < n; r++) {
      const double w = W[r];
      s += (w * ai[r]) * (w * aj[r]);
    }
    Accumulate(G + (long)j * ldg + i, s, acc);
  });
  t.par(m, [&](int j) {
    const double* aj = Ac + (long)j * n;
    double aw = 0, aq = 0;
    for (int r = 0; r < n; r++) {
      const double w = W[r];
      aw += aj[r] * w;
      aq += (w * aj[r]) * (w * c[r]);
    }
    Accumulate(AW + j, aw, acc);
    Accumulate(AQc + j, aq, acc);
  });
  const double s1 = t.sum(n, [&](int r) { return W[r] * c[r]; });
  const double s2 = t.sum(n, [&](int r) {
    const double v = W[r] * c[r];
    return v * v;
  });
  t.single([&]() {
    Accumulate(scal + 0, s1, acc);
    Accumulate(scal + 1, s2, acc);
  });
}

// out4 = {lambda_min, lambda_max, frobenius_norm_squared, trace} (linear_constraint.cc:148-166)
template <class T>
CXB_HD void LpEigen(T& t, int n, int m, const double* Ac, const double* y, double cw, const double* W,
                    double* t1, double* t2, double* out4) {
  NegativeSlack(t, n, m, Ac, y, cw, t1);
  t.par(n, [&](int r) { t2[r] = W[r] * t1[r]; });
  const double mn = t.minv(n, [&](int r) { return t2[r]; });
  const double mx = t.maxv(n, [&](int r) { return t2[r]; });
  const double sq = t.sum(n, [&](int r) { return t2[r] * t2[r]; });
  const double sm = t.sum(n, [&](int r) { return t2[r]; });
  t.single([&]() {
    out4[0] = -mx;
    out4[1] = -mn;
    out4[2] = sq;
    out4[3] = -sm;
  });
}

// out2 = {norminfd, normsqrd} (linear_constraint.cc:108-129, affine branch :174-179)
template <class T>
CXB_HD void LpPrepare(T& t, int n, int m, const double* Ac, const double* y, bool affine, double cw,
                      double ew, double* W, double* t1, double* t2, double* out2) {
  if (!affine) {
    NegativeSlack(t, n, m, Ac, y, cw, t2);
    t.par(n, [&](int r) { t2[r] = t2[r] * W[r] + ew; });
    const double ninf = t.maxv(n, [&](int r) { return fabs(t2[r]); });
    const double nsq = t.sum(n, [&](int r) { return t2[r] * t2[r]; });
    t.single([&]() {
      out2[0] = ninf;
      out2[1] = nsq;
    });
  } else {
    NegativeSlack(t, n, m, Ac, y, 0.0, t1);
    t.par(n, [&](int r) {
      const double sw = t1[r] * W[r];
      t1[r] = sw;
      W[r] += W[r] * sw;
    });
    t.single([&]() {
      out2[0] = 0;
      out2[1] = 0;
    });
  }
}

// W <- W .* exp(step * d), d = t2 (linear_constraint.cc:131-145)
template <class T>
CXB_HD void LpTakeStep(T& t, int n, double step, double* W, double* t2) {
  t.par(n, [&](int r) {
    double d = t2[r];
    if (step != 1.0) d *= step;
    d = exp(d);
    t2[r] = d;
    W[r] *= d;
  });
}

// =================================================================================================
// Second-order cone of order o = n + 1 (spin factor). state: Wv[o] = (W0, W1), d[o].
// work: o * (m + 1) + 3 * o doubles.
// =================================================================================================
// out = f(ev0) c0 + f(ev1) c1 with the spectral decomposition of x (soc_constraint.cc:22-63,131-170);
// fn: 0 sqrt, 1 exp. out must not alias x.
template <class T>
CXB_HD void SpinFunction(T& t, int o, const double* x, int fn, double* out) {
  const double nq = sqrt(t.sum(o - 1, [&](int i) { return x[1 + i] * x[1 + i]; }));
  const double e0 = x[0] + nq, e1 = x[0] - nq;
  const double f0 = fn ? exp(e0) : sqrt(e0);
  const double f1 = fn ? exp(e1) : sqrt(e1);
  t.par(o, [&](int i) {
    if (i == 0) {
      out[0] = f0 * .5 + f1 * .5;
    } else {
      const double q = (nq > 0) ? x[i] / nq : 0.0;
      out[i] = f0 * (.5 * q) + f1 * (-.5 * q);
    }
  });
}

// det x = x0^2 - |x1|^2
template <class T>
CXB_HD double SpinDet(T& t, int o, const double* x) {
  return x[0] * x[0] - t.sum(o - 1, [&](int i) { return x[1 + i] * x[1 + i]; });
}

// out = Q(x) y = 2 <x, y> x - det(x) R y (soc_constraint.cc:115-128); serial, one thread.
CXB_HD void QuadRepSerial(int o, const double* x, double det, const double* y, double* out) {
  double xy = 0;
  for (int i = 0; i < o; i++) xy += x[i] * y[i];
  for (int i = 0; i < o; i++) {
    double z = det * y[i];
    if (i == 0) z *= -1;
    out[i] = (2 * xy) * x[i] + z;
  }
}
// Same by the whole team; out must not alias x or y.
template <class T>
CXB_HD void QuadRep(T& t, int o, const double* x, const double* y, double* out) {
  const double det = SpinDet(t, o, x);
  const double xy = t.sum(o, [&](int i) { return x[i] * y[i]; });
  t.par(o, [&](int i) {
    double z = det * y[i];
    if (i == 0) z *= -1;
    out[i] = (2 * xy) * x[i] + z;
  });
}

template <class T>
CXB_HD void SocSetIdentity(T& t, int o, double* Wv) {
  t.par(o, [&](int i) { Wv[i] = (i == 0) ? 1.0 : 0.0; });
}

template <class T>
CXB_HD void SocSchur(T& t, int o, int m, const double* Ac, const double* Wv, double* work, double* G,
                     long ldg, double* AW, double* AQc, double* scal, bool acc) {
  double* wsqrt = work;
  double* WA = work + o;  // o x (m + 1); column m = Q(w^{1/2}) c
  SpinFunction(t, o, Wv, 0, wsqrt);
  const double det = SpinDet(t, o, wsqrt);
  t.par(m + 1, [&](int j) { QuadRepSerial(o, wsqrt, det, Ac + (long)j * o, WA + (long)j * o); });
  const double* WC = WA + (long)m * o;
  const Divider by_m(m);
  t.par(m * m, [&](int e) {
    const int j = by_m.quot(e), i = e - j * m;
    if (i < j) return;
    double s = 0;
    for (int r = 0; r < o; r++) s += WA[(long)i * o + r] * WA[(long)j * o + r];
    Accumulate(G + (long)j * ldg + i, 2 * s, acc);
  });
  t.par(m, [&](int j) {
    double aw = 0, aq = 0;
    for (int r = 0; r < o; r++) {
      aw += Ac[(long)j * o + r] * Wv[r];
      aq += WA[(long)j * o + r] * WC[r];
    }
    Accumulate(AW + j, 2 * aw, acc);
    Accumulate(AQc + j, 2 * aq, acc);
  });
  const double sq = t.sum(o, [&](int r) { return WC[r] * WC[r]; });
  t.single([&]() {
    Accumulate(scal + 0, 2 * WC[0], acc);
    Accumulate(scal + 1, 2 * sq, acc);
  });
}

template <class T>
CXB_HD void SocEigen(T& t, int o, int m, const double* Ac, const double* y, double cw, const double* Wv,
                     double* work, double* out4) {
  double* minus_s = work;
  double* wsqrt = work + o;
  double* Ws = work + 2 * o;
  NegativeSlack(t, o, m, Ac, y, cw, minus_s);
  SpinFunction(t, o, Wv, 0, wsqrt);
  QuadRep(t, o, wsqrt, minus_s, Ws);
  const double nq = sqrt(t.sum(o - 1, [&](int i) { return Ws[1 + i] * Ws[1 + i]; }));
  t.single([&]() {
    const double ev0 = Ws[0] + nq, ev1 = Ws[0] - nq;
    const double lmax = -fmin(ev0, ev1), lmin = -fmax(ev0, ev1);
    out4[0] = lmin;
    out4[1] = lmax;
    out4[2] = lmax * lmax + lmin * lmin;
    out4[3] = lmax + lmin;
  });
}

// NB (soc_constraint.cc:213-230): W is replaced by its square root, e_weight / affine are ignored.
template <class T>
CXB_HD void SocPrepare(T& t, int o, int m, const double* Ac, const double* y, double cw, double* Wv,
                       double* d, double* work, double* out2) {
  double* minus_s = work;
  double* wsqrt = work + o;
  NegativeSlack(t, o, m, Ac, y, cw, minus_s);
  SpinFunction(t, o, Wv, 0, wsqrt);
  QuadRep(t, o, wsqrt, minus_s, d);
  t.par(o, [&](int i) {
    Wv[i] = wsqrt[i];
    if (i == 0) d[0] += 1;
  });
  const double nq = sqrt(t.sum(o - 1, [&](int i) { return d[1 + i] * d[1 + i]; }));
  const double sq = t.sum(o, [&](int i) { return d[i] * d[i]; });
  t.single([&]() {
    out2[0] = fmax(fabs(d[0] + nq), fabs(d[0] - nq));
    out2[1] = 2 * sq;
  });
}

// W <- Q(w^{1/2}) exp(step * d)  (soc_constraint.cc:191-211; Wv already holds w^{1/2})
template <class T>
CXB_HD void SocTakeStep(T& t, int o, double step, double* Wv, const double* d, double* work) {
  double* ds = work;
  double* expd = work + o;
  double* wn = work + 2 * o;
  t.par(o, [&](int i) { ds[i] = (step != 1.0) ? d[i] * step : d[i]; });
  SpinFunction(t, o, ds, 1, expd);
  QuadRep(t, o, Wv, expd, wn);
  t.par(o, [&](int i) { Wv[i] = wn[i]; });
}

// =================================================================================================
// Small dense PSD / LMI block of order n (n*n doubles per matrix fit in shared memory).
// state: W, T1, T2 (n*n each, global). sm: shared scratch of 6 n*n + 8 n + 16 doubles.
// work (global): (m + 2) n*n doubles for the scaled matrices W A_i W, W C W and a copy of W.
// =================================================================================================
// C = A * B (n x n, column-major, all three distinct)
template <class T>
CXB_HD void MatMul(T& t, int n, const double* A, const double* B, double* C) {
  if ((n & 1) == 0) {
    // 2 x 2 outputs per thread: four loads feed four FMAs per k (one output per thread: two loads per FMA, and these
    // products are issue-bound). Every output is the same sum in the same order.
    const int h = n / 2;
    const Divider by_h(h);
    t.par(h * h, [&](int e) {
      const int c2 = by_h.quot(e), r2 = e - c2 * h;
      const int r = 2 * r2, c = 2 * c2;
      double s00 = 0, s10 = 0, s01 = 0, s11 = 0;
      for (int k = 0; k < n; k++) {
        const double a0 = A[k * n + r], a1 = A[k * n + r + 1];
        const double b0 = B[c * n + k], b1 = B[(c + 1) * n + k];
        s00 += a0 * b0;
        s10 += a1 * b0;
        s01 += a0 * b1;
        s11 += a1 * b1;
      }
      C[c * n + r] = s00;
      C[c * n + r + 1] = s10;
      C[(c + 1) * n + r] = s01;
      C[(c + 1) * n + r + 1] = s11;
    });
    return;
  }
  const Divider by_n(n);
  t.par(n * n, [&](int e) {
    const int c = by_n.quot(e), r = e - c * n;
    double s = 0;
    for (int k = 0; k < n; k++) s += A[k * n + r] * B[c * n + k];
    C[e] = s;
  });
}

template <class T>
CXB_HD void PsdSetIdentity(T& t, int n, double* W) {
  t.par(n * n, [&](int e) { W[e] = (e % (n + 1) == 0) ? 1.0 : 0.0; });
}

// H_ij = <W A_i W, A_j> (lower), AW_j = <W, A_j>, AQc_j = <W C W, A_j>, <w,c> = <W, C>,
// <c,Qc> = <W C W, C>  (dense_lmi_constraint.cc:62-103).
//
// Phase A scales the matrices, B_i = W (A_i W), `group` matrices at a time with 4 x 4 register tiles
// (per k: two 4-vectors from shared memory feed 16 FMAs); T = A_i W is kept row-major so that both
// operands of the second product are contiguous. Phase B is the Gram contraction C = B^T A over the
// n^2 entries (an (m+2) x (m+1) x n^2 GEMM, lower tiles only) with 4 x 2 register tiles, the
// operands staged through shared memory in chunks of kGramChunk entries (coalesced global reads)
// and the accumulators parked in shared memory between chunks.
// work (global): (m + 2) n^2 doubles. sm: PsdSchurSmemDoubles(n, m, team size) doubles.
constexpr int kGramChunk = 40;
CXB_HOST_DEVICE int PsdSchurGroup(int n, int team) {
  const int tn = (n + 3) / 4;
  const int g = team / (tn * tn);
  return g < 1 ? 1 : g;
}
CXB_HOST_DEVICE long PsdSchurSmemDoubles(int n, int m, int team) {
  const long nn = (long)n * n;
  const long a = nn + 2 * PsdSchurGroup(n, team) * nn;
  const long ti = (m + 2 + 3) / 4, tj = (m + 1 + 1) / 2;
  const long b = (long)(2 * m + 3) * (kGramChunk + 1) + ti * tj * 8;
  // symmetric form: W -> L and L^T (2 nn), then `group` matrices and their products (2 group nn)
  const long c = 2 * nn + 2 * PsdSchurGroup(n, team) * nn;
  const long ab = a > b ? a : b;
  return ab > c ? ab : c;
}

template <class T>
CXB_HD void PsdSchurClassic(T& t, int n, int m, const double* AC, const double* W, double* work, double* sm,
                            double* G, long ldg, double* AW, double* AQc, double* scal, bool acc) {
  const int nn = n * n;
  const int tn = (n + 3) / 4, tiles = tn * tn;
  const int group = PsdSchurGroup(n, t.size());
  // ---- phase A ---------------------------------------------------------------------------------------
  {
    double* sW = sm;
    double* sA = sm + nn;
    double* sT = sA + (long)group * nn;
    t.par(nn, [&](int e) { sW[e] = W[e]; });
    for (int i0 = 0; i0 <= m; i0 += group) {
      const int gc = (m + 1 - i0 < group) ? m + 1 - i0 : group;
      const double* src = AC + (long)i0 * nn;
      t.par(gc * nn, [&](int e) { sA[e] = src[e]; });
      // T = A W, stored row-major: sT[r * n + c]. W is symmetric: W[k][c] = sW[k * n + c].
      t.par(gc * tiles, [&](int w) {
        const int g = w / tiles, tile = w % tiles;
        const int r0 = (tile % tn) * 4, c0 = (tile / tn) * 4;
        const double* A = sA + (long)g * nn;
        double c[4][4] = {{0, 0, 0, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}};
        for (int k = 0; k < n; k++) {
          double a[4], b[4];
#pragma unroll
          for (int x = 0; x < 4; x++) a[x] = (r0 + x < n) ? A[k * n + r0 + x] : 0.0;
#pragma unroll
          for (int y = 0; y < 4; y++) b[y] = (c0 + y < n) ? sW[k * n + c0 + y] : 0.0;
#pragma unroll
          for (int x = 0; x < 4; x++)
#pragma unroll
            for (int y = 0; y < 4; y++) c[x][y] += a[x] * b[y];
        }
        double* Tg = sT + (long)g * nn;
#pragma unroll
        for (int x = 0; x < 4; x++)
#pragma unroll
          for (int y = 0; y < 4; y++)
            if (r0 + x < n && c0 + y < n) Tg[(r0 + x) * n + c0 + y] = c[x][y];
      });
      // B = W T -> global work (column-major)
      t.par(gc * tiles, [&](int w) {
        const int g = w / tiles, tile = w % tiles;
        const int r0 = (tile % tn) * 4, c0 = (tile / tn) * 4;
        const double* Tg = sT + (long)g * nn;
        double c[4][4] = {{0, 0, 0, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}};
        for (int k = 0; k < n; k++) {
          double a[4], b[4];
#pragma unroll
          for (int x = 0; x < 4; x++) a[x] = (r0 + x < n) ? sW[k * n + r0 + x] : 0.0;
#pragma unroll
          for (int y = 0; y < 4; y++) b[y] = (c0 + y < n) ? Tg[k * n + c0 + y] : 0.0;
#pragma unroll
          for (int x = 0; x < 4; x++)
#pragma unroll
            for (int y = 0; y < 4; y++) c[x][y] += a[x] * b[y];
        }
        double* Bg = work + (long)(i0 + g) * nn;
#pragma unroll
        for (int y = 0; y < 4; y++)
#pragma unroll
          for (int x = 0; x < 4; x++)
            if (r0 + x < n && c0 + y < n) Bg[(c0 + y) * n + r0 + x] = c[x][y];
      });
    }
    t.par(nn, [&](int e) { work[(long)(m + 1) * nn + e] = sW[e]; });  // row m + 1 of the Gram: W itself
  }
  // ---- phase B ---------------------------------------------------------------------------------------
  const int MI = m + 2, MJ = m + 1;
  const int ti = (MI + 3) / 4, tj = (MJ + 1) / 2;
  const int P = kGramChunk + 1;
  double* sB = sm;
  double* sAc = sm + (long)MI * P;
  double* sAcc = sAc + (long)MJ * P;
  t.par(ti * tj * 8, [&](int e) { sAcc[e] = 0.0; });
  for (int q0 = 0; q0 < nn; q0 += kGramChunk) {
    const int kc = (nn - q0 < kGramChunk) ? nn - q0 : kGramChunk;
    t.par((MI + MJ) * kc, [&](int e) {
      const int row = e / kc, q = e % kc;
      if (row < MI) {
        sB[row * P + q] = work[(long)row * nn + q0 + q];
      } else {
        sAc[(row - MI) * P + q] = AC[(long)(row - MI) * nn + q0 + q];
      }
    });
    t.par(ti * tj, [&](int w) {
      const int i0 = (w % ti) * 4, j0 = (w / ti) * 2;
      if (i0 + 3 < j0) return;  // tile entirely above the diagonal
      double c[4][2];
#pragma unroll
      for (int x = 0; x < 4; x++) {
        c[x][0] = sAcc[w * 8 + 2 * x];
        c[x][1] = sAcc[w * 8 + 2 * x + 1];
      }
      const double* b0 = sB + (long)(i0 + 0 < MI ? i0 + 0 : MI - 1) * P;
      const double* b1 = sB + (long)(i0 + 1 < MI ? i0 + 1 : MI - 1) * P;
      const double* b2 = sB + (long)(i0 + 2 < MI ? i0 + 2 : MI - 1) * P;
      const double* b3 = sB + (long)(i0 + 3 < MI ? i0 + 3 : MI - 1) * P;
      const double* a0 = sAc + (long)(j0 + 0 < MJ ? j0 + 0 : MJ - 1) * P;
      const double* a1 = sAc + (long)(j0 + 1 < MJ ? j0 + 1 : MJ - 1) * P;
      for (int q = 0; q < kc; q++) {
        const double x0 = b0[q], x1 = b1[q], x2 = b2[q], x3 = b3[q], y0 = a0[q], y1 = a1[q];
        c[0][0] += x0 * y0;
        c[0][1] += x0 * y1;
        c[1][0] += x1 * y0;
        c[1][1] += x1 * y1;
        c[2][0] += x2 * y0;
        c[2][1] += x2 * y1;
        c[3][0] += x3 * y0;
        c[3][1] += x3 * y1;
      }
#pragma unroll
      for (int x = 0; x < 4; x++) {
        sAcc[w * 8 + 2 * x] = c[x][0];
        sAcc[w * 8 + 2 * x + 1] = c[x][1];
      }
    });
  }
  t.par(ti * tj * 8, [&](int e) {
    const int w = e / 8, x = (e % 8) / 2, y = e % 2;
    const int i = (w % ti) * 4 + x, j = (w / ti) * 2 + y;
    if (i >= MI || j >= MJ || i < j) return;
    const double s = sAcc[e];
    if (i < m) {
      Accumulate(G + (long)j * ldg + i, s, acc);
    } else if (i == m) {
      Accumulate(j < m ? AQc + j : scal + 1, s, acc);
    } else {
      Accumulate(j < m ? AW + j : scal + 0, s, acc);
    }
  });
}

// The same Schur system from the symmetric form (DESIGN.md 3.1, here for one small block): with
// W = L L^T, H_ij = <L^T A_i L, L^T A_j L>, so phase A forms S_i = L^T (A_i L) — the first product skips
// the zeros above L's diagonal, the second computes lower tiles only: 1.33 n^3 instead of 4 n^3 per
// matrix — and stores only its lower triangle, off-diagonal entries scaled by sqrt(2) so that the plain
// dot product of two packed matrices is their trace inner product; phase B is then X X^T over
// n (n + 1) / 2 entries instead of n^2, with both operands read from the same array. The packed
// identity stands in for W in the row that yields AW_j = tr(W A_j) = <I, S_j>.
// Returns false (nothing written) when W is not numerically positive definite; the caller then uses
// the classic form, which needs no factorisation.
template <class T>
CXB_HD bool PsdSchurSymmetric(T& t, int n, int m, const double* AC, const double* W, double* work, double* sm,
                              double* G, long ldg, double* AW, double* AQc, double* scal, bool acc) {
  const int nn = n * n;
  const int kp = n * (n + 1) / 2;
  const int tn = (n + 3) / 4, tiles = tn * tn;
  const int group = PsdSchurGroup(n, t.size());
  const double kSqrt2 = 1.4142135623730951;
  // ---- L = chol(W): sL column-major (zeros above the diagonal), sLT its transpose --------------------
  double* sL = sm;
  double* sLT = sm + nn;
  t.par(nn, [&](int e) { sL[e] = (e % n >= e / n) ? W[e] : 0.0; });
  for (int j = 0; j < n; j++) {
    const double d = sL[j * n + j];  // same value in every thread (barrier at the end of the last phase)
    if (!(d > 0.0)) return false;
    const int rem = n - j - 1;
    t.par(rem * rem, [&](int e) {
      const int r = j + 1 + e % rem, c = j + 1 + e / rem;
      if (r >= c) sL[c * n + r] -= sL[j * n + r] * sL[j * n + c] / d;
    });
    const double rd = sqrt(d);
    t.par(n - j, [&](int i) { sL[j * n + j + i] = (i == 0) ? rd : sL[j * n + j + i] / rd; });
  }
  t.par(nn, [&](int e) { sLT[(e % n) * n + e / n] = sL[e]; });  // sLT[k * n + c] = L(k, c)
  // ---- phase A: S_i = L^T (A_i L), lower triangle, packed ---------------------------------------------
  {
    double* sA = sm + 2 * nn;
    double* sT = sA + (long)group * nn;
    for (int i0 = 0; i0 <= m; i0 += group) {
      const int gc = (m + 1 - i0 < group) ? m + 1 - i0 : group;
      const double* src = AC + (long)i0 * nn;
      t.par(gc * nn, [&](int e) { sA[e] = src[e]; });
      // T = A L, row-major sT[r * n + c]; L(k, c) = 0 for k < c: the k loop starts at the tile's column
      t.par(gc * tiles, [&](int w) {
        const int g = w / tiles, tile = w % tiles;
        const int r0 = (tile % tn) * 4, c0 = (tile / tn) * 4;
        const double* A = sA + (long)g * nn;
        double c[4][4] = {{0, 0, 0, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}};
        for (int k = c0; k < n; k++) {
          double a[4], b[4];
#pragma unroll
          for (int x = 0; x < 4; x++) a[x] = (r0 + x < n) ? A[k * n + r0 + x] : 0.0;
#pragma unroll
          for (int y = 0; y < 4; y++) b[y] = (c0 + y < n) ? sLT[k * n + c0 + y] : 0.0;
#pragma unroll
          for (int x = 0; x < 4; x++)
#pragma unroll
            for (int y = 0; y < 4; y++) c[x][y] += a[x] * b[y];
        }
        double* Tg = sT + (long)g * nn;
#pragma unroll
        for (int x = 0; x < 4; x++)
#pragma unroll
          for (int y = 0; y < 4; y++)
            if (r0 + x < n && c0 + y < n) Tg[(r0 + x) * n + c0 + y] = c[x][y];
      });
      // S = L^T T, tiles on or below the diagonal only; L^T(r, k) = L(k, r) = 0 for k < r
      t.par(gc * tiles, [&](int w) {
        const int g = w / tiles, tile = w % tiles;
        const int r0 = (tile % tn) * 4, c0 = (tile / tn) * 4;
        if (r0 + 3 < c0) return;
        const double* Tg = sT + (long)g * nn;
        double c[4][4] = {{0, 0, 0, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}};
        for (int k = r0; k < n; k++) {
          double a[4], b[4];
#pragma unroll
          for (int x = 0; x < 4; x++) a[x] = (r0 + x < n) ? sLT[k * n + r0 + x] : 0.0;
#pragma unroll
          for (int y = 0; y < 4; y++) b[y] = (c0 + y < n) ? Tg[k * n + c0 + y] : 0.0;
#pragma unroll
          for (int x = 0; x < 4; x++)
#pragma unroll
            for (int y = 0; y < 4; y++) c[x][y] += a[x] * b[y];
        }
        double* Sg = work + (long)(i0 + g) * kp;
#pragma unroll
        for (int y = 0; y < 4; y++)
#pragma unroll
          for (int x = 0; x < 4; x++) {
            const int r = r0 + x, cc = c0 + y;
            if (r < n && cc <= r) Sg[cc * n - cc * (cc - 1) / 2 + (r - cc)] = (r == cc) ? c[x][y] : kSqrt2 * c[x][y];
          }
      });
    }
    // row m + 1: the packed identity
    t.par(nn, [&](int e) {
      const int r = e % n, cc = e / n;
      if (cc <= r) work[(long)(m + 1) * kp + cc * n - cc * (cc - 1) / 2 + (r - cc)] = (r == cc) ? 1.0 : 0.0;
    });
  }
  // ---- phase B: Gram of the packed matrices -----------------------------------------------------------
  const int MI = m + 2, MJ = m + 1;
  const int ti = (MI + 3) / 4, tj = (MJ + 1) / 2;
  const int P = kGramChunk + 1;
  double* sB = sm;
  double* sAcc = sm + (long)MI * P;
  t.par(ti * tj * 8, [&](int e) { sAcc[e] = 0.0; });
  for (int q0 = 0; q0 < kp; q0 += kGramChunk) {
    const int kc = (kp - q0 < kGramChunk) ? kp - q0 : kGramChunk;
    t.par(MI * kc, [&](int e) {
      const int row = e / kc, q = e % kc;
      sB[row * P + q] = work[(long)row * kp + q0 + q];
    });
    t.par(ti * tj, [&](int w) {
      const int i0 = (w % ti) * 4, j0 = (w / ti) * 2;
      if (i0 + 3 < j0) return;  // tile entirely above the diagonal
      double c[4][2];
#pragma unroll
      for (int x = 0; x < 4; x++) {
        c[x][0] = sAcc[w * 8 + 2 * x];
        c[x][1] = sAcc[w * 8 + 2 * x + 1];
      }
      const double* b0 = sB + (long)(i0 + 0 < MI ? i0 + 0 : MI - 1) * P;
      const double* b1 = sB + (long)(i0 + 1 < MI ? i0 + 1 : MI - 1) * P;
      const double* b2 = sB + (long)(i0 + 2 < MI ? i0 + 2 : MI - 1) * P;
      const double* b3 = sB + (long)(i0 + 3 < MI ? i0 + 3 : MI - 1) * P;
      const double* a0 = sB + (long)(j0 + 0 < MJ ? j0 + 0 : MJ - 1) * P;
      const double* a1 = sB + (long)(j0 + 1 < MJ ? j0 + 1 : MJ - 1) * P;
      for (int q = 0; q < kc; q++) {
        const double x0 = b0[q], x1 = b1[q], x2 = b2[q], x3 = b3[q], y0 = a0[q], y1 = a1[q];
        c[0][0] += x0 * y0;
        c[0][1] += x0 * y1;
        c[1][0] += x1 * y0;
        c[1][1] += x1 * y1;
        c[2][0] += x2 * y0;
        c[2][1] += x2 * y1;
        c[3][0] += x3 * y0;
        c[3][1] += x3 * y1;
      }
#pragma unroll
      for (int x = 0; x < 4; x++) {
        sAcc[w * 8 + 2 * x] = c[x][0];
        sAcc[w * 8 + 2 * x + 1] = c[x][1];
      }
    });
  }
  t.par(ti * tj * 8, [&](int e) {
    const int w = e / 8, x = (e % 8) / 2, y = e % 2;
    const int i = (w % ti) * 4 + x, j = (w / ti) * 2 + y;
    if (i >= MI || j >= MJ || i < j) return;
    const double s = sAcc[e];
    if (i < m) {
      Accumulate(G + (long)j * ldg + i, s, acc);
    } else if (i == m) {
      Accumulate(j < m ? AQc + j : scal + 1, s, acc);
    } else {
      Accumulate(j < m ? AW + j : scal + 0, s, acc);
    }
  });
  return true;
}

// form: 0 = symmetric when W factors, else classic (default); 1 = classic (the reference's formula).
template <class T>
CXB_HD void PsdSchur(T& t, int n, int m, const double* AC, const double* W, double* work, double* sm,
                     double* G, long ldg, double* AW, double* AQc, double* scal, bool acc, int form = 0) {
  if (form == 0 && PsdSchurSymmetric(t, n, m, AC, W, work, sm, G, ldg, AW, AQc, scal, acc)) return;
  PsdSchurClassic(t, n, m, AC, W, work, sm, G, ldg, AW, AQc, scal, acc);
}

// Extreme eigenvalues of the symmetric tridiagonal (alpha[0..k), beta[0..k-1)) by Sturm bisection —
// device twin of host/tridiagonal_eigenvalues.cc (the reference takes min/max of the full spectrum,
// approximate_eigenvalues.cc:235-237). Serial.
CXB_HD int SturmCountBelow(const double* a, const double* b, int k, double x, double tiny) {
  int count = 0;
  double q = 1;
  for (int i = 0; i < k; i++) {
    const double off = (i == 0) ? 0.0 : (b[i - 1] * b[i - 1]) / q;
    q = a[i] - x - off;
    if (fabs(q) < tiny) q = -tiny;
    if (q < 0) count++;
  }
  return count;
}
CXB_HD double SturmKth(const double* a, const double* b, int k, int which, double lo, double hi,
                       double tiny) {
  for (int it = 0; it < 200; it++) {
    const double mid = 0.5 * (lo + hi);
    if (mid <= lo || mid >= hi) break;
    if (SturmCountBelow(a, b, k, mid, tiny) > which) {
      hi = mid;
    } else {
      lo = mid;
    }
  }
  return 0.5 * (lo + hi);
}
CXB_HD void ExtremeTridiagonal(const double* a, const double* b, int k, double* emin, double* emax) {
  if (k == 1) {
    *emin = *emax = a[0];
    return;
  }
  const double eps = 2.220446049250313e-16;
  double lo = 1.7976931348623157e308, hi = -1.7976931348623157e308, scale = 0;
  for (int i = 0; i < k; i++) {
    const double r = (i > 0 ? fabs(b[i - 1]) : 0.0) + (i + 1 < k ? fabs(b[i]) : 0.0);
    lo = fmin(lo, a[i] - r);
    hi = fmax(hi, a[i] + r);
    scale = fmax(scale, fabs(a[i]) + r);
  }
  const double pad = 4 * eps * (scale + 1e-300) * (double)k;
  lo -= pad;
  hi += pad;
  double tiny = 2.2250738585072014e-308 / eps + 1e-30 * scale * scale;
  tiny = fmax(tiny, eps * eps * scale);
  *emin = SturmKth(a, b, k, 0, lo, hi, tiny);
  *emax = SturmKth(a, b, k, k - 1, lo, hi, tiny);
}

// The same two eigenvalues by multi-section with the whole team: every round evaluates the Sturm count at
// kSections interior points of a bracket at once (one point per thread) and keeps the sub-interval that still holds the
// wanted eigenvalue — the first point whose count exceeds `which`, found with a team-wide first_true (a ballot in the
// warp layout) — so a bracket shrinks by kSections + 1 per round (11 rounds to full double precision) instead of by 2
// per serial bisection step. The brackets are uniform values held in registers by every thread: a round is one phase
// per bracket, with no serial section. (The first version selected the sub-interval in a single-thread loop over the
// kSections counts — 2 x 32 dependent shared-memory reads and divisions per round, more than the Sturm counts
// themselves and the largest part of the batched eigen-bound kernels.) Converges to the same eigenvalues as
// ExtremeTridiagonal up to the final bracket width. `scratch` is unused (kept for the callers' layout).
constexpr int kSections = 32;
template <class T>
CXB_HD void ExtremeTridiagonalTeam(T& t, const double* a, const double* b, int k, double* scratch, double* emin,
                                   double* emax) {
  (void)scratch;
  if (k == 1) {
    t.single([&]() { *emin = *emax = a[0]; });
    return;
  }
  // Gershgorin bounds: every thread computes the same values (k <= n / 2 entries)
  const double eps = 2.220446049250313e-16;
  double lo = 1.7976931348623157e308, hi = -1.7976931348623157e308, scale = 0;
  for (int i = 0; i < k; i++) {
    const double r = (i > 0 ? fabs(b[i - 1]) : 0.0) + (i + 1 < k ? fabs(b[i]) : 0.0);
    lo = fmin(lo, a[i] - r);
    hi = fmax(hi, a[i] + r);
    scale = fmax(scale, fabs(a[i]) + r);
  }
  const double pad = 4 * eps * (scale + 1e-300) * (double)k;
  lo -= pad;
  hi += pad;
  double tiny = 2.2250738585072014e-308 / eps + 1e-30 * scale * scale;
  tiny = fmax(tiny, eps * eps * scale);
  double result[2];
  for (int side = 0; side < 2; side++) {
    const int which = side == 0 ? 0 : k - 1;
    double l = lo, h = hi;
    for (int round = 0; round < 64; round++) {
      const double w = h - l;
      const double first = l + w * (1.0 / (double)(kSections + 1));
      const double last = l + w * ((double)kSections / (double)(kSections + 1));
      if (!(first > l) || !(last < h)) break;  // the interior points no longer resolve the bracket: converged
      const int q = t.first_true(kSections, [&](int i) {
        const double x = l + w * ((double)(i + 1) / (double)(kSections + 1));
        return SturmCountBelow(a, b, k, x, tiny) > which;
      });
      const double nl = q == 0 ? l : l + w * ((double)q / (double)(kSections + 1));
      const double nh = q == kSections ? h : l + w * ((double)(q + 1) / (double)(kSections + 1));
      l = nl;
      h = nh;
    }
    result[side] = 0.5 * (l + h);
  }
  t.single([&]() {
    *emin = result[0];
    *emax = result[1];
  });
}

// Two-sided Lanczos on (WS, WS^T) in the W inner product started from r
// (approximate_eigenvalues.cc:178-239, num_iter = n/2, breakdown beta^2 < 1e-6), then the extreme
// Ritz values. vec: 6 n + 2 (n/2 + 2) doubles of scratch. Returns through ritz[0..1].
template <class T>
CXB_HD void LanczosExtremes(T& t, int n, const double* WS, const double* W, const double* r, double* vec,
                            double* ritz) {
  double *v0 = vec, *v1 = vec + n, *u0 = vec + 2 * n, *u1 = vec + 3 * n, *p0 = vec + 4 * n,
         *p1 = vec + 5 * n;
  double* alpha = vec + 6 * n;
  double* beta = alpha + n / 2 + 2;
  const int num_iter = n / 2;
  if (n == 1 || num_iter < 1) {  // ApproximateEigenvalues returns WS itself (:248-250)
    t.single([&]() { ritz[0] = ritz[1] = WS[0]; });
    return;
  }
  t.par(n, [&](int i) {
    double s = 0;
    for (int k = 0; k < n; k++) s += W[k * n + i] * r[k];
    v0[i] = s;
    v1[i] = r[i];
  });
  const double scale = sqrt(t.sum(n, [&](int i) { return v0[i] * v1[i]; }));
  t.par(n, [&](int i) {
    v0[i] /= scale;
    v1[i] /= scale;
  });
  int count = 0;
  double bprev = 0;
  for (int j = 0; j < num_iter; j++) {
    t.par(n, [&](int i) {
      double a0 = 0, a1 = 0;
      for (int k = 0; k < n; k++) {
        a0 += WS[k * n + i] * v0[k];  // (WS v0)[i]
        a1 += WS[i * n + k] * v1[k];  // (WS^T v1)[i]
      }
      u0[i] = a0;
      u1[i] = a1;
    });
    const double a = t.sum(n, [&](int i) { return v0[i] * u1[i]; });
    t.par(n, [&](int i) {
      double x0 = u0[i] - a * v0[i], x1 = u1[i] - a * v1[i];
      if (j > 0) {
        x0 -= bprev * p0[i];
        x1 -= bprev * p1[i];
      }
      u0[i] = x0;
      u1[i] = x1;
    });
    const double b2 = t.sum(n, [&](int i) { return u0[i] * u1[i]; });
    t.single([&]() { alpha[j] = a; });
    count = j;
    if (j + 1 >= num_iter || b2 < 1e-6) break;
    const double bj = sqrt(b2);
    t.par(n, [&](int i) {
      p0[i] = v0[i];
      p1[i] = v1[i];
      v0[i] = u0[i] / bj;
      v1[i] = u1[i] / bj;
    });
    t.single([&]() { beta[j] = bj; });
    bprev = bj;
  }
  ExtremeTridiagonalTeam(t, alpha, beta, count + 1, beta + n / 2 + 2, ritz + 0, ritz + 1);
}

// S -> T1, WS = W S -> T2 (global state) and shared copies; returns tr(WS), tr(WS WS) and the
// index of the largest diagonal entry of WS (first occurrence).
// sm layout: sW | sS | sWS | vec...
// packed (may be null): the lower triangles of the matrices of AC (symmetric matrices: same sums, half the reads).
template <class T>
CXB_HD void PsdWeightedSlack(T& t, int n, int m, const double* AC, const double* packed, const double* y, double cw,
                             const double* W, double* T1, double* T2, double* sm, double* trace,
                             double* trace_sq, int* index) {
  const int nn = n * n;
  double* sW = sm;
  double* sS = sm + nn;
  double* sWS = sm + 2 * nn;
  t.par(nn, [&](int e) { sW[e] = W[e]; });
  if (packed != nullptr) {
    double* sP = sWS;  // n (n + 1) / 2 doubles, free until the product below
    NegativeSlack(t, n * (n + 1) / 2, m, packed, y, cw, sP);
    const Divider by_rows(n);
    t.par(nn, [&](int e) {
      const int c = by_rows.quot(e), r = e - c * n;
      const int lo = r < c ? r : c, hi = r < c ? c : r;  // entry (hi, lo) of the lower triangle
      sS[e] = sP[lo * n - lo * (lo - 1) / 2 + (hi - lo)];
    });
  } else {
    NegativeSlack(t, nn, m, AC, y, cw, sS);
  }
  MatMul(t, n, sW, sS, sWS);
  t.par(nn, [&](int e) {
    T1[e] = sS[e];
    T2[e] = sWS[e];
  });
  *trace = t.sum(n, [&](int i) { return sWS[i * n + i]; });
  const Divider by_n(n);
  *trace_sq = t.sum(nn, [&](int e) {
    const int c = by_n.quot(e), r = e - c * n;
    return sWS[e] * sWS[r * n + c];
  });
  double largest;
  *index = t.argmax_first(n, [&](int i) { return sWS[i * n + i]; }, &largest);
}

// out4 = {lambda_min, lambda_max, frobenius_norm_squared, trace} (psd_constraint.cc:97-128)
template <class T>
CXB_HD void PsdEigen(T& t, int n, int m, const double* AC, const double* y, double cw, const double* W,
                     double* T1, double* T2, double* sm, double* out4, const double* packed = nullptr) {
  const int nn = n * n;
  double tr, trsq;
  int index;
  PsdWeightedSlack(t, n, m, AC, packed, y, cw, W, T1, T2, sm, &tr, &trsq, &index);
  double* ritz = sm + 3 * nn;
  // start vector: column `index` of the true -S
  t.warp0([&](auto& w) { LanczosExtremes(w, n, sm + 2 * nn, sm, sm + nn + index * n, sm + 3 * nn + 2, ritz); });
  t.single([&]() {
    out4[0] = -ritz[1];
    out4[1] = -ritz[0];
    out4[2] = trsq;
    out4[3] = -tr;
  });
}

// out2 = {norminfd, normsqrd} (psd_constraint.cc:45-84); affine: W <- (1 + ew) W + (W S) W (:33-43)
template <class T>
CXB_HD void PsdPrepare(T& t, int n, int m, const double* AC, const double* y, bool affine, double cw,
                       double ew, double* W, double* T1, double* T2, double* sm, double* out2,
                       const double* packed = nullptr) {
  const int nn = n * n;
  double tr, trsq;
  int index;
  PsdWeightedSlack(t, n, m, AC, packed, y, cw, W, T1, T2, sm, &tr, &trsq, &index);
  if (affine) {
    double* sT = sm + nn;  // the slack is no longer needed
    MatMul(t, n, sm + 2 * nn, sm, sT);
    t.par(nn, [&](int e) {
      double w = sm[e];
      if (ew != 0.0) w *= (1.0 + ew);
      W[e] = w + sT[e];
    });
    t.single([&]() {
      out2[0] = 0;
      out2[1] = 0;
    });
    return;
  }
  double* ritz = sm + 3 * nn;
  // the reference starts from a column of WS here (minus_s aliases WS, psd_constraint.cc:48-69)
  t.warp0([&](auto& w) { LanczosExtremes(w, n, sm + 2 * nn, sm, sm + 2 * nn + index * n, sm + 3 * nn + 2, ritz); });
  t.single([&]() {
    out2[0] = fmax(fabs(ew + ritz[0]), fabs(ew + ritz[1]));
    out2[1] = trsq + 2 * tr + n;
  });
}

// W <- sym( pade33( step (WS + ew I) ) W ), WS = T2 (psd_constraint.cc:13-28,
// exponential_map_pade.cc:10-32). sm: 6 n*n doubles. info: set to 1 + column on a zero pivot.
template <class T>
CXB_HD void PsdTakeStep(T& t, int n, double step, double ew, double* W, const double* T2, double* sm,
                        int* info) {
  const int nn = n * n;
  double* X = sm;
  double* X2 = sm + nn;
  double* U = sm + 2 * nn;
  double* M = sm + 3 * nn;  // n x 2n: [V - U | V + U]
  double* sW = sm + 5 * nn;
  const Divider by_n(n), by_diag(n + 1);  // e is a diagonal entry iff e % (n + 1) == 0
  t.par(nn, [&](int e) {
    X[e] = (T2[e] + ((by_diag.rem(e) == 0) ? ew : 0.0)) * step;
    sW[e] = W[e];
  });
  MatMul(t, n, X, X, X2);
  t.par(nn, [&](int e) { M[e] = X2[e] + ((by_diag.rem(e) == 0) ? 60.0 : 0.0); });
  MatMul(t, n, X, M, U);  // U = X (X^2 + 60 I)
  t.par(nn, [&](int e) {
    const double v = 12.0 * X2[e] + ((by_diag.rem(e) == 0) ? 120.0 : 0.0);
    const double u = U[e];
    M[e] = v - u;
    M[nn + e] = v + u;
  });
  // Gaussian elimination with partial (row) pivoting on the n x 2n augmented matrix
  for (int k = 0; k < n; k++) {
    // pivot = the first entry of largest magnitude in column k, rows k..n-1 (a team reduction instead of a serial
    // scan by one thread: 20 dependent shared-memory reads per column were a third of this function's chain)
    double bv;
    const int p = k + t.argmax_first(n - k, [&](int i) { return fabs(M[k * n + k + i]); }, &bv);
    if (bv == 0.0) t.single([&]() { if (*info == 0) *info = k + 1; });
    if (p != k) {
      t.par(2 * n, [&](int c) {
        const double tmp = M[c * n + k];
        M[c * n + k] = M[c * n + p];
        M[c * n + p] = tmp;
      });
    }
    // One phase per column: rows on lanes, columns on warps; the multiplier of a row is computed by every thread that
    // needs it and is not stored (the back substitution below only reads the upper triangle and the right-hand sides).
    const double piv = M[k * n + k];
    t.par2(
        n - k - 1, 2 * n - k - 1, [&](int i) { return M[k * n + k + 1 + i] / piv; },
        [&](int i, int c, double l) { M[(k + 1 + c) * n + k + 1 + i] -= l * M[(k + 1 + c) * n + k]; });
  }
  // back substitution, one right-hand-side column per thread
  t.par(n, [&](int c) {
    double* b = M + nn + c * n;
    for (int i = n - 1; i >= 0; i--) {
      double s = b[i];
      for (int k = i + 1; k < n; k++) s -= M[k * n + i] * b[k];
      b[i] = s / M[i * n + i];
    }
  });
  MatMul(t, n, M + nn, sW, X);  // E W
  t.par(nn, [&](int e) {
    const int c = by_n.quot(e), r = e - c * n;
    W[e] = 0.5 * (X[e] + X[r * n + c]);
  });
}

// =================================================================================================
// Small dense KKT system (N x N lower, ld): Cholesky in shared memory and the two triangular solves.
// =================================================================================================
// sH: N*N doubles of shared memory. info: 0 or 1 + column of the first non-positive pivot.
template <class T>
CXB_HD void SmallPotrf(T& t, int N, double* H, long ld, double* sH, int* info) {
  const Divider by_N(N);
  t.par(N * N, [&](int e) {
    const int c = by_N.quot(e), r = e - c * N;
    sH[e] = (r >= c) ? H[(long)c * ld + r] : 0.0;
  });
  int failed = 0;
  for (int j = 0; j < N; j++) {
    // The diagonal keeps the pivot d_j until the end (every thread reads it here, so nobody may
    // overwrite it in this phase); its square root is taken in one sweep after the loop.
    const double d = sH[j * N + j];
    if (!(d > 0.0)) {
      failed = j + 1;
      break;
    }
    const double rd = sqrt(d);
    t.par(N - j - 1, [&](int i) { sH[j * N + j + 1 + i] /= rd; });
    const int w = N - j - 1;
    t.par2(
        w, w, [&](int i) { return sH[j * N + j + 1 + i]; },
        [&](int i, int c, double lr) {
          if (i >= c) sH[(j + 1 + c) * N + j + 1 + i] -= lr * sH[j * N + j + 1 + c];
        });
  }
  if (failed) {
    t.single([&]() { *info = failed; });
    return;
  }
  t.par(N * N, [&](int e) {
    const int c = by_N.quot(e), r = e - c * N;
    if (r > c) H[(long)c * ld + r] = sH[e];
    if (r == c) H[(long)c * ld + r] = sqrt(sH[e]);
  });
  t.single([&]() { *info = 0; });
}

// x <- L^{-T} L^{-1} x. sx: N doubles shared.
template <class T>
CXB_HD void SmallPotrs(T& t, int N, const double* L, long ld, double* x, double* sx) {
  t.par(N, [&](int i) { sx[i] = x[i]; });
  for (int j = 0; j < N; j++) {
    // sx[j] is final here and is not written in this phase (it is divided by L_jj afterwards)
    const double xj = sx[j] / L[(long)j * ld + j];
    t.par(N - j - 1, [&](int i) { sx[j + 1 + i] -= L[(long)j * ld + j + 1 + i] * xj; });
  }
  t.par(N, [&](int j) { sx[j] /= L[(long)j * ld + j]; });
  for (int j = N - 1; j >= 0; j--) {
    const double s = t.sum(N - j - 1, [&](int i) { return L[(long)j * ld + j + 1 + i] * sx[j + 1 + i]; });
    t.single([&]() { sx[j] = (sx[j] - s) / L[(long)j * ld + j]; });
  }
  t.par(N, [&](int i) { x[i] = sx[i]; });
}

// =================================================================================================
// Small KKT system with equality multipliers (N = variables + multipliers, symmetric indefinite): the regularised
// LDL^T of Eigen::RLDLT (RLDLT.h:297-431) as L S L^T, S = diag(+-1), |D|^{1/2} folded into L — the arithmetic of
// cxb_sym_permute_lower + cxb_ldlt_lower (cholesky.cu, LdltDiagKernel) for one program, in shared memory.
// =================================================================================================
// The pivot that Eigen::RLDLT's left-looking algorithm takes at step k is the largest |d| among positions k.. of
// the CURRENT arrangement (lowest position on ties), swapped to position k; those entries are still the original
// diagonal, so the whole order follows from diag(K) (host RldltPivotOrder, cone_program.cc). A selection with
// swaps, not a stable sort. One warp: a shuffle arg-max per step. sd: the N |d| (shared, permuted in place);
// at[i]: original index at position i.
template <class W>
CXB_HD void RldltPivotOrder(W& w, int N, double* sd, int* at) {
  for (int k = 0; k + 1 < N; k++) {
    double v;
    const int p = k + w.argmax_first(N - k, [&](int i) { return sd[k + i]; }, &v);
    if (p != k) {
      w.single([&]() {
        const double d = sd[k];
        sd[k] = sd[p];
        sd[p] = d;
        const int a = at[k];
        at[k] = at[p];
        at[p] = a;
      });
    }
  }
}

// A pivot with |d| <= 1e-9 is used as -1e-9 when d < 0 and as +1e-9 otherwise (RLDLT.h:378-389).
CXB_HD double RegularisedPivot(double d) { return (fabs(d) > 1e-9) ? d : ((d < 0) ? -1e-9 : 1e-9); }

// K (N x N, lower triangle read, ld ldk) is not modified. Writes the lower triangle of L (ldl), perm[i] = original
// index at pivot position i and signs = S; returns 1 when some pivot was regularised, else 0 (it never fails).
// sH: N*N doubles, sd: N doubles, at: N ints, all shared.
template <class T>
CXB_HD int SmallLdlt(T& t, int N, const double* K, long ldk, double* L, long ldl, int* perm, double* signs,
                     double* sH, double* sd, int* at) {
  t.par(N, [&](int i) {
    sd[i] = fabs(K[(long)i * ldk + i]);
    at[i] = i;
  });
  t.warp0([&](auto& w) { RldltPivotOrder(w, N, sd, at); });
  // P K P^T from the lower triangle of K, the permutation fused into the load
  const Divider by_N(N);
  t.par(N * N, [&](int e) {
    const int c = by_N.quot(e), r = e - c * N;
    if (r >= c) {
      const int i = at[r], j = at[c];
      sH[e] = (i >= j) ? K[(long)j * ldk + i] : K[(long)i * ldk + j];
    }
  });
  int regularised = 0;
  for (int j = 0; j < N; j++) {
    // the diagonal keeps the (unregularised) pivot until the end, as in SmallPotrf
    double d = sH[j * N + j];
    if (!(fabs(d) > 1e-9)) regularised = 1;
    d = RegularisedPivot(d);
    const double sign = (d < 0) ? -1.0 : 1.0;
    const double inv = 1.0 / sqrt(fabs(d));
    // column j of L = sign a_j / sqrt|d|; the update of entry (r, c) is sign a_r a_c / |d| = L_rj (sign L_cj)
    t.par(N - j - 1, [&](int i) { sH[j * N + j + 1 + i] *= sign * inv; });
    const int w = N - j - 1;
    t.par2(
        w, w, [&](int i) { return sH[j * N + j + 1 + i]; },
        [&](int i, int c, double lr) {
          if (i >= c) sH[(j + 1 + c) * N + j + 1 + i] -= lr * (sign * sH[j * N + j + 1 + c]);
        });
  }
  t.par(N * N, [&](int e) {
    const int c = by_N.quot(e), r = e - c * N;
    if (r > c) L[(long)c * ldl + r] = sH[e];
    if (r == c) {
      const double d = RegularisedPivot(sH[e]);
      L[(long)c * ldl + r] = sqrt(fabs(d));
      signs[r] = (d < 0) ? -1.0 : 1.0;
      perm[r] = at[r];
    }
  });
  return regularised;
}

// x <- P^T L^{-T} S L^{-1} P x with the factors of SmallLdlt. sx: N doubles shared.
template <class T>
CXB_HD void SmallLdltSolve(T& t, int N, const double* L, long ld, const int* perm, const double* signs, double* x,
                           double* sx) {
  t.par(N, [&](int i) { sx[i] = x[perm[i]]; });
  for (int j = 0; j < N; j++) {
    const double xj = sx[j] / L[(long)j * ld + j];
    t.par(N - j - 1, [&](int i) { sx[j + 1 + i] -= L[(long)j * ld + j + 1 + i] * xj; });
  }
  t.par(N, [&](int j) { sx[j] = signs[j] * (sx[j] / L[(long)j * ld + j]); });
  for (int j = N - 1; j >= 0; j--) {
    const double s = t.sum(N - j - 1, [&](int i) { return L[(long)j * ld + j + 1 + i] * sx[j + 1 + i]; });
    t.single([&]() { sx[j] = (sx[j] - s) / L[(long)j * ld + j]; });
  }
  t.par(N, [&](int i) { x[perm[i]] = sx[i]; });
}

// =================================================================================================
// KKT systems whose N x N matrix does not fit in shared memory (cxb_small_potrf / cxb_small_ldlt above the sizes of
// SmallPotrf / SmallLdlt): the same two factorisations, blocked and right-looking, in place in global memory. Per
// block column of kKktNb columns: the diagonal block is factored in shared memory with the per-column arithmetic of
// SmallPotrf / SmallLdlt; the panel below it is solved one row per thread (the row in registers, the block's
// columns in sequence); the trailing matrix takes A22 -= L21 S L21^T on its lower triangle (`update`: the DMMA tiles
// of small_cones.cu on the device, KktTrailingUpdateLoop on the host). The scratch does not depend on N.
// =================================================================================================
constexpr int kKktNb = 32;
constexpr int kKktPitch = kKktNb + 1;  // odd pitch of the diagonal block
// sm: the diagonal block, then per column the scale (Cholesky: sqrt(d); LDL^T: sign / sqrt|d|) and the sign
CXB_HOST_DEVICE long BlockedKktSmemDoubles() { return (long)kKktNb * kKktPitch + 2 * kKktNb; }

// A22 -= L21 S L21^T on the lower triangle: the trailing R x R matrix at (t0, t0) of A, L21 = the kb columns from k0
// of its rows, S = s[0..kb). Plain team loop; the product's kernels use DMMA tiles instead.
struct KktTrailingUpdateLoop {
  template <class T>
  CXB_HD void operator()(T& t, double* A, long ld, int k0, int kb, int t0, int R, const double* s) const {
    const Divider by_R(R);
    t.par(R * R, [&](int e) {
      const int c = by_R.quot(e), r = e - c * R;
      if (r < c) return;
      double acc = 0;
      for (int k = 0; k < kb; k++) {
        const double* col = A + (long)(k0 + k) * ld + t0;
        acc += col[r] * (s[k] * col[c]);
      }
      A[(long)(t0 + c) * ld + t0 + r] -= acc;
    });
  }
};

// The factorisation of A (N x N lower, ld) in place. LDLT == false: Cholesky; returns 0, or 1 + the first column
// whose pivot is not > 0 (A is then left partly factored). LDLT == true: the regularised L S L^T of SmallLdlt, S
// written to signs; returns 1 when some pivot was regularised, else 0. Either way the diagonal keeps the
// (unregularised) pivot until its block column is done, then stores sqrt|reg(d)|.
template <bool LDLT, class T, class U>
CXB_HD int BlockedFactor(T& t, int N, double* A, long ld, double* signs, double* sm, const U& update) {
  constexpr int P = kKktPitch;
  double* sD = sm;
  double* sScale = sm + kKktNb * P;
  double* sSign = sScale + kKktNb;
  int regularised = 0;
  for (int k0 = 0; k0 < N; k0 += kKktNb) {
    const int kb = (N - k0 < kKktNb) ? N - k0 : kKktNb;
    double* Ak = A + (long)k0 * ld + k0;  // the diagonal block
    t.par(kb * kb, [&](int e) {
      const int c = e / kb, r = e - c * kb;
      if (r >= c) sD[c * P + r] = Ak[(long)c * ld + r];
    });
    for (int j = 0; j < kb; j++) {
      double d = sD[j * P + j];
      double sign = 1.0;
      if (LDLT) {
        if (!(fabs(d) > 1e-9)) regularised = 1;
        d = RegularisedPivot(d);
        sign = (d < 0) ? -1.0 : 1.0;
      } else if (!(d > 0.0)) {
        return k0 + j + 1;  // d is the same in every thread
      }
      const double scale = LDLT ? sign * (1.0 / sqrt(fabs(d))) : sqrt(d);
      t.par(kb - j, [&](int i) {
        if (i == 0) {
          sScale[j] = scale;
          sSign[j] = sign;
        } else if (LDLT) {
          sD[j * P + j + i] *= scale;
        } else {
          sD[j * P + j + i] /= scale;
        }
      });
      const int w = kb - j - 1;
      t.par2(
          w, w, [&](int i) { return sD[j * P + j + 1 + i]; },
          [&](int i, int c, double lr) {
            if (i >= c) sD[(j + 1 + c) * P + j + 1 + i] -= lr * (sign * sD[j * P + j + 1 + c]);
          });
    }
    t.par(kb * kb, [&](int e) {
      const int c = e / kb, r = e - c * kb;
      if (r > c) Ak[(long)c * ld + r] = sD[c * P + r];
      if (r == c) {
        const double d = LDLT ? RegularisedPivot(sD[c * P + r]) : sD[c * P + r];
        Ak[(long)c * ld + r] = sqrt(fabs(d));
        if (LDLT) signs[k0 + r] = (d < 0) ? -1.0 : 1.0;
      }
    });
    // the panel: row i of L21 = row i of A21 solved against the block's columns, the same steps as its entries take
    // in SmallPotrf / SmallLdlt once the earlier blocks' updates are in
    const int t0 = k0 + kb, R = N - t0;
    if (R == 0) break;
    t.par(R, [&](int i) {
      double* row = A + (long)k0 * ld + t0 + i;  // entry (t0 + i, k0 + c) at row[c * ld]
      double x[kKktNb];
#pragma unroll
      for (int c = 0; c < kKktNb; c++) x[c] = (c < kb) ? row[(long)c * ld] : 0.0;
#pragma unroll
      for (int j = 0; j < kKktNb; j++) {
        if (j < kb) {
          x[j] = LDLT ? x[j] * sScale[j] : x[j] / sScale[j];
          const double sj = sSign[j];
#pragma unroll
          for (int c = j + 1; c < kKktNb; c++)
            if (c < kb) x[c] -= x[j] * (sj * sD[j * P + c]);
        }
      }
#pragma unroll
      for (int c = 0; c < kKktNb; c++)
        if (c < kb) row[(long)c * ld] = x[c];
    });
    update(t, A, ld, k0, kb, t0, R, sSign);
  }
  return LDLT ? regularised : 0;
}

// Cholesky of H (N x N lower, ld) in place: 0, or 1 + the first column whose pivot is not > 0 (H is then
// unspecified). sm: BlockedKktSmemDoubles() doubles.
template <class T, class U>
CXB_HD int BlockedPotrf(T& t, int N, double* H, long ld, double* sm, const U& update) {
  return BlockedFactor<false>(t, N, H, ld, nullptr, sm, update);
}

// SmallLdlt without the N x N shared copy: the pivot order of RldltPivotOrder (warp 0), P K P^T gathered from the
// lower triangle of K straight into L, then L factored in place. K is not modified. sm: BlockedKktSmemDoubles()
// doubles; sd: N doubles, at: N ints (shared).
template <class T, class U>
CXB_HD int BlockedLdlt(T& t, int N, const double* K, long ldk, double* L, long ldl, int* perm, double* signs,
                       double* sm, double* sd, int* at, const U& update) {
  t.par(N, [&](int i) {
    sd[i] = fabs(K[(long)i * ldk + i]);
    at[i] = i;
  });
  t.warp0([&](auto& w) { RldltPivotOrder(w, N, sd, at); });
  const Divider by_N(N);
  t.par(N * N, [&](int e) {
    const int c = by_N.quot(e), r = e - c * N;
    if (r >= c) {
      const int i = at[r], j = at[c];
      L[(long)c * ldl + r] = (i >= j) ? K[(long)j * ldk + i] : K[(long)i * ldk + j];
    }
  });
  t.par(N, [&](int i) { perm[i] = at[i]; });
  return BlockedFactor<true>(t, N, L, ldl, signs, sm, update);
}

}  // namespace small
}  // namespace cxb

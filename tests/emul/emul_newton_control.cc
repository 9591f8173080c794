// TEST INFRASTRUCTURE ONLY — never linked into libconex_b200.so.
//
// A C interface to the host-only NewtonControl (conex_b200/csrc/host/newton_control.cc) for
// tests/test_newton_control.py, compiled with it and divergence.cc by g++.
#include <cstddef>

#include "newton_control.h"
#include "divergence.h"

using conex::NewtonControl;
using conex::SolverConfiguration;
using conex::WeightedSlackEigenvalues;

namespace {

// the configuration fields NewtonControl reads, in the order of nc_fields()
#define NC_FIELDS(X)                                                                                                  \
  X(initialization_mode) X(inv_sqrt_mu_max) X(maximum_mu) X(divergence_upper_bound) X(enable_line_search)            \
  X(final_centering_steps) X(final_centering_tolerance) X(initial_centering_steps_warmstart)                         \
  X(initial_centering_steps_coldstart) X(warmstart_abort_threshold) X(max_iterations) X(infeasibility_threshold)      \
  X(kkt_error_tolerance) X(enable_rescaling)

struct Handle {
  SolverConfiguration cfg;  // NewtonControl keeps a pointer to it
  NewtonControl control;
  Handle(const SolverConfiguration& c, int rank, const double* b, int n, double bs, double cs)
      : cfg(c), control(cfg, rank, b, static_cast<size_t>(n), bs, cs) {}
};

NewtonControl& C(void* h) { return static_cast<Handle*>(h)->control; }

WeightedSlackEigenvalues Summary(double lmin, double lmax, double frob, double trace) {
  WeightedSlackEigenvalues w;
  w.lambda_min = lmin;
  w.lambda_max = lmax;
  w.frobenius_norm_squared = frob;
  w.trace = trace;
  return w;
}

}  // namespace

extern "C" {

const char* nc_fields() {
#define NC_NAME(f) #f ","
  return NC_FIELDS(NC_NAME);
#undef NC_NAME
}

void nc_default_config(double* v) {
  SolverConfiguration c;
  int j = 0;
#define NC_GET(f) v[j++] = static_cast<double>(c.f);
  NC_FIELDS(NC_GET)
#undef NC_GET
}

void* nc_create(const double* v, int rank, const double* b, int n, double b_scaling, double c_scaling) {
  SolverConfiguration c;
  int j = 0;
#define NC_SET(f) c.f = static_cast<decltype(c.f)>(v[j++]);
  NC_FIELDS(NC_SET)
#undef NC_SET
  return new Handle(c, rank, b, n, b_scaling, c_scaling);
}

void nc_destroy(void* h) { delete static_cast<Handle*>(h); }

int nc_begin(void* h, int i) { return C(h).Begin(i); }
int nc_needs_aqc_norm(void* h) { return C(h).NeedsAqcNorm(); }
void nc_rescale(void* h, double aqc_norm_squared) { C(h).Rescale(aqc_norm_squared); }
int nc_restart_on_factorization_failure(void* h) { return C(h).RestartOnFactorizationFailure(); }
int nc_update_mu(void* h) { return C(h).update_mu(); }
int nc_needs_eigenvalues(void* h) { return C(h).NeedsEigenvalues(); }

// cones: ncones x {lambda_min, lambda_max, frobenius_norm_squared, trace}, reduced as both drivers reduce them
void nc_choose_k(void* h, int ncones, const double* cones) {
  conex::SlackEigenvalueSum w;
  for (int k = 0; k < ncones; k++) w.Add(cones[4 * k], cones[4 * k + 1], cones[4 * k + 2], cones[4 * k + 3]);
  C(h).ChooseK(w);
}

int nc_step(void* h, double norminfd, double normsqrd, double* step_size) {
  return C(h).Step(norminfd, normsqrd, step_size);
}

int nc_end(void* h, double b_dot_y, double aqc_dot_y, double w_dot_c, double c_dot_qc) {
  return C(h).End(b_dot_y, aqc_dot_y, w_dot_c, c_dot_qc);
}

// status: solved, num_iterations, primal_infeasible, dual_infeasible
void nc_finish(void* h, double* y, int n, int* status) {
  const conex::ConexStatus s = C(h).Finish(y, static_cast<size_t>(n));
  status[0] = s.solved;
  status[1] = s.num_iterations;
  status[2] = s.primal_infeasible;
  status[3] = s.dual_infeasible;
}

// k, mu, b_scaling, c_scaling, by, cx, kkt_error, d_2, d_inf | num_iterations, stepping, failed
void nc_state(void* h, double* d, int* flags) {
  const NewtonControl& c = C(h);
  const double v[] = {c.k(), c.mu(), c.b_scaling(), c.c_scaling(), c.by(), c.cx(), c.kkt_error(), c.d_2(), c.d_inf()};
  for (int j = 0; j < 9; j++) d[j] = v[j];
  flags[0] = c.num_iterations();
  flags[1] = c.stepping();
  flags[2] = c.failed();
}

void nc_scale_dual_variable(int num_iterations, int primal_infeasible, double inv_sqrt_mu, double b_scaling,
                            double* w, int n) {
  conex::ScaleDualVariable(num_iterations, primal_infeasible, inv_sqrt_mu, b_scaling, w, static_cast<size_t>(n));
}

double nc_divergence_upper_bound_inverse(double bound, double lmin, double lmax, double frob, double trace,
                                         double rank) {
  WeightedSlackEigenvalues w = Summary(lmin, lmax, frob, trace);
  w.rank = rank;
  return conex::DivergenceUpperBoundInverse(bound, w);
}

}  // extern "C"

// The per-program control of the interior-point loop (reference cone_program.cc:235-533): centering schedule,
// rescaling, mu rule, step size, warm-start aborts, objectives, convergence and status; host code only.
// NewtonDriver::Run keeps one instance and BatchProgram::Maximize one per program, which launch the kernels that
// produce the inputs: per iteration Begin, Rescale, (RestartOnFactorizationFailure,) ChooseK, Step, End; then Finish.
#pragma once
#include "cone_program.h"

namespace conex {

class NewtonControl {
 public:
  // b: the cost (n entries); rank: the cones' ranks summed; b/c_scaling: the last solve's, which a warm start keeps
  NewtonControl(const SolverConfiguration& cfg, int rank, const double* b, size_t n, double b_scaling,
                double c_scaling);

  bool Begin(int i);  // false: the solve has ended
  // iteration 0 with rescaling on: a cold start takes |AQc|^2 (read when NeedsAqcNorm()) and |b| as new scalings
  bool NeedsAqcNorm() const { return i_ == 0 && cfg_->enable_rescaling && !warm_; }
  void Rescale(double aqc_norm_squared);
  // true: a warm start restarts, the cones are reset to the identity and the iteration ends; false: the solve fails
  bool RestartOnFactorizationFailure();
  bool update_mu() const { return update_mu_; }
  bool NeedsEigenvalues() const { return update_mu_ && LineSearchCandidate() < 0; }
  // w: the slack eigenvalues at H^{-1}(AQc c_scaling - b b_scaling), read when NeedsEigenvalues()
  void ChooseK(const WeightedSlackEigenvalues& w);
  // The norms of the direction, reduced over the cones as PrepareStep reports them (reference
  // cone_program.cc:418-436). Sets *step_size; false: reset the cones to the identity instead of stepping.
  bool Step(double norminfd, double normsqrd, double* step_size);
  // b.y, AQc.y, <w,c>, <c,Qc> after the step (reference cone_program.cc:441-478); true: converged.
  bool End(double b_dot_y, double aqc_dot_y, double w_dot_c, double c_dot_qc);
  // The status (reference cone_program.cc:486-530); y (n entries) /= k c_scaling unless infeasible or failed.
  ConexStatus Finish(double* y, size_t n) const;

  // false once stopped at Begin, converged or failed to factor, and in an iteration restarted by a warm start
  bool stepping() const { return !done_ && !restarted_; }
  bool failed() const { return failed_; }
  double k() const { return k_; }
  double mu() const { return (1.0 / k_) * (1.0 / k_) / (c_scaling_ * b_scaling_); }
  double b_scaling() const { return b_scaling_; }
  double c_scaling() const { return c_scaling_; }
  double by() const { return by_; }
  double cx() const { return cx_; }
  double kkt_error() const { return kkt_error_; }
  double d_2() const { return d_2_; }
  double d_inf() const { return d_inf_; }
  int num_iterations() const { return num_iter_; }

 private:
  // PSD / second-order cones provide no PerformLineSearch (reference constraint.h:24-28): the search fails and k is
  // kept (cone_program.cc:376-384). The drivers refuse line search on programs of LP cones only.
  double LineSearchCandidate() const { return cfg_->enable_line_search ? k_ : -1; }
  double MuFromEigenvalues(WeightedSlackEigenvalues p) const;

  const SolverConfiguration* cfg_;
  bool warm_;
  int rank_;
  int initial_centering_steps_;
  int i_ = -1;
  double k_ = 0, kmax_, cx_ = 1, by_ = -1, kkt_error_ = 0;
  double b_scaling_, c_scaling_, b_norm_ = 0, d_2_ = 0, d_inf_ = 0;
  int centering_steps_ = 0, num_iter_ = 0;
  bool done_ = false, failed_ = false, max_iters_reached_ = true, warmstart_aborted_ = false;
  bool initial_centering_ = false, final_centering_ = false, update_mu_ = false;
  bool restarted_ = false;  // this iteration: the warm start failed to factor, the cones were reset
};

// The program's summary from its cones' (reference cone_program.cc:31-57), from lambda_min / lambda_max = +-30000.
struct SlackEigenvalueSum : WeightedSlackEigenvalues {
  SlackEigenvalueSum() { lambda_min = 30000; lambda_max = -30000; }
  void Add(double cone_lambda_min, double cone_lambda_max, double cone_frobenius_norm_squared, double cone_trace);
};

// A cone's dual variable as a solve reports it: W / (k b_scaling) at the last iterate (reference
// cone_program.h:120-134); W as it is after a solve without iterations or a primal infeasible one.
void ScaleDualVariable(int num_iterations, int primal_infeasible, double inv_sqrt_mu, double b_scaling, double* w,
                       size_t n);

}  // namespace conex

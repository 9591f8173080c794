#include "newton_control.h"

#include <algorithm>
#include <cmath>

#include "divergence.h"

namespace conex {

NewtonControl::NewtonControl(const SolverConfiguration& cfg, int rank, const double* b, size_t n, double b_scaling,
                             double c_scaling)
    : cfg_(&cfg),
      warm_(cfg.initialization_mode != CONEX_INITIALIZATION_MODE_COLDSTART),
      rank_(rank),
      initial_centering_steps_(warm_ ? cfg.initial_centering_steps_warmstart : cfg.initial_centering_steps_coldstart),
      kmax_(cfg.inv_sqrt_mu_max),
      b_scaling_(b_scaling),
      c_scaling_(c_scaling) {
  for (size_t j = 0; j < n; j++) b_norm_ += b[j] * b[j];
  b_norm_ = std::sqrt(b_norm_);
}

// reference cone_program.cc:312-336
bool NewtonControl::Begin(int i) {
  if (done_) return false;
  i_ = i;
  restarted_ = false;
  initial_centering_ = i < initial_centering_steps_;
  final_centering_ = (k_ >= kmax_) || (kkt_error_ > cfg_->kkt_error_tolerance) ||
                     (i >= cfg_->max_iterations - cfg_->final_centering_steps);
  update_mu_ = (i == 0) || !(initial_centering_ || final_centering_) || warmstart_aborted_;
  warmstart_aborted_ = false;
  if (final_centering_ && centering_steps_ >= cfg_->final_centering_steps) {
    max_iters_reached_ = (i >= cfg_->max_iterations - 1);
    done_ = true;
    return false;
  }
  return true;
}

// reference cone_program.cc:343-357: a cold start takes new scalings, a warm start keeps those of the previous solve
void NewtonControl::Rescale(double aqc_norm_squared) {
  if (i_ != 0 || !cfg_->enable_rescaling) return;
  if (!warm_) {
    b_scaling_ = 1.0 / (1 + b_norm_);
    c_scaling_ = 1.0 / (1 + std::sqrt(aqc_norm_squared));
  }
  // xhat*shat = mu I for the scaled iterates means x*s = mu/(b_scaling*c_scaling): rescale the target.
  const double mu_target = (1.0 / (kmax_ * kmax_)) * (b_scaling_ * c_scaling_);
  kmax_ = 1.0 / std::sqrt(mu_target);
}

// reference cone_program.cc:360-371: only the first factorisation of a warm start may fail without failing the solve
bool NewtonControl::RestartOnFactorizationFailure() {
  restarted_ = warmstart_aborted_ = i_ == 0 && warm_;
  done_ = failed_ = !restarted_;
  return restarted_;
}

// reference cone_program.cc:166-214
double NewtonControl::MuFromEigenvalues(WeightedSlackEigenvalues p) const {
  p.rank = rank_;
  double k = DivergenceUpperBoundInverse(cfg_->divergence_upper_bound * rank_, p);
  if (k == -1) {
    // maximise the denominator of the bound instead (cone_program.cc:166-172)
    k = (p.lambda_min > 0) ? 2.0 / (p.lambda_min + p.lambda_max) : -1;
  }
  if (k < 0 && p.trace > 1e-12) {
    // last resort: the mu that satisfies a norm bound (cone_program.cc:194-211)
    const double kstar = p.trace / p.frobenius_norm_squared;
    double norm_bound = 1.5 * (p.frobenius_norm_squared * kstar * kstar - 2 * p.trace * kstar + rank_);
    norm_bound = std::min(norm_bound, rank_ * .7);
    const double qa = p.frobenius_norm_squared, qb = -2 * p.trace, qc = rank_ - norm_bound;
    const double disc = qb * qb - 4 * qa * qc;
    k = (disc < 0) ? kstar : (-qb + std::sqrt(disc)) / (2 * qa);
  }
  return k;
}

// reference cone_program.cc:373-399
void NewtonControl::ChooseK(const WeightedSlackEigenvalues& w) {
  if (update_mu_) {
    double candidate = LineSearchCandidate();
    if (candidate < 0) candidate = MuFromEigenvalues(w);
    k_ = (candidate > 0) ? candidate : 0.5 * k_;
  } else if (!initial_centering_) {
    centering_steps_++;
  }
  k_ = std::max(std::min(k_, kmax_), std::sqrt(1.0 / (1e-15 + cfg_->maximum_mu)));
}

bool NewtonControl::Step(double norminfd, double normsqrd, double* step_size) {
  d_2_ = std::sqrt(std::fabs(normsqrd));
  d_inf_ = std::fabs(norminfd);
  *step_size = std::min(1.0, 2.0 / (norminfd * norminfd));
  if (i_ == 0 && warm_ && norminfd >= cfg_->warmstart_abort_threshold) {
    // too large a first step from the warm iterate: the cones restart from the identity; the iteration still counts
    warmstart_aborted_ = true;
    return false;
  }
  return true;
}

bool NewtonControl::End(double b_dot_y, double aqc_dot_y, double w_dot_c, double c_dot_qc) {
  by_ = b_dot_y / (k_ * c_scaling_);
  // k <c,x> = 2 <c,w> + <AQc, y> - k <c,Qc>   (reference cone_program.cc:443-452)
  cx_ = (2 * w_dot_c + aqc_dot_y - k_ * c_dot_qc * c_scaling_) / (k_ * b_scaling_);
  const double mu = (1.0 / k_) * (1.0 / k_);
  const double s_dot_x = mu * (rank_ - d_2_ * d_2_) / (b_scaling_ * c_scaling_);
  kkt_error_ = std::fabs(cx_ - by_ - s_dot_x) / s_dot_x;
  num_iter_ = i_ + 1;
  if ((final_centering_ || k_ >= kmax_) && d_inf_ <= cfg_->final_centering_tolerance) {
    max_iters_reached_ = false;
    done_ = true;
  }
  return done_;
}

ConexStatus NewtonControl::Finish(double* y, size_t n) const {
  ConexStatus status;
  status.num_iterations = num_iter_;
  if (failed_) return status;
  if ((1.0 / k_) * (1.0 / k_) > cfg_->infeasibility_threshold) {  // mu_final
    status.primal_infeasible = cx_ * k_ <= -.5;
    status.dual_infeasible = by_ * k_ >= .5;
    return status;
  }
  for (size_t j = 0; j < n; j++) y[j] = y[j] / k_ / c_scaling_;
  status.solved = !max_iters_reached_;
  return status;
}

void SlackEigenvalueSum::Add(double cone_lambda_min, double cone_lambda_max, double cone_frobenius_norm_squared,
                             double cone_trace) {
  lambda_max = std::max(lambda_max, cone_lambda_max);
  lambda_min = std::min(lambda_min, cone_lambda_min);
  frobenius_norm_squared += cone_frobenius_norm_squared;
  trace += cone_trace;
}

void ScaleDualVariable(int num_iterations, int primal_infeasible, double inv_sqrt_mu, double b_scaling, double* w,
                       size_t n) {
  if (primal_infeasible || num_iterations <= 0) return;
  const double scale = inv_sqrt_mu * b_scaling;
  for (size_t j = 0; j < n; j++) w[j] /= scale;
}

}  // namespace conex

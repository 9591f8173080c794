// Many small, structurally identical cone programs advanced in lock step on one GPU — the
// "batched small-block SDP" regime (BASELINE config 3; SURVEY.md §8e: independent units, no
// collective). The reference solves such programs one after the other on the CPU, each through
// Solve() (conex/cone_program.cc:235-533); distinct Program handles are independent
// (interfaces/conex.cc has no shared state), which is what makes batching legal.
//
// Design: the cone data of all B programs is packed cone by cone into batched device arrays; every
// phase of the Newton step is ONE launch per cone with one CTA per program (device/small_cones.cu),
// the B small KKT systems are factored and solved by one launch each, and the per-program control
// flow of Solve() — centering schedule, mu rule, rescaling, step size, termination, status — runs on
// the host over arrays of B scalars fetched once per phase, in one NewtonControl per program
// (newton_control.h), the class that also drives a single program's solve. Programs that have
// terminated are masked out of later launches, so every program follows exactly the iteration
// sequence it would follow alone.
//
// Equality constraints (EqualityConstraints blocks, on any subset of the variables) add their
// multipliers as KKT unknowns m..N-1, in the order the blocks were added (Program::AddConstraint).
// Their rows of the KKT matrices and of AQc / AW are constant and written once per batch; the cones'
// Schur kernels assign only the leading m x m block. A batch with multipliers factors its KKT systems
// with the batched regularised LDL^T (cxb_small_ldlt, never fails), one without keeps the batched
// Cholesky — the input decides, as in kkt_solver.cc:172-199. Both take any KKT order N: the device
// layer factors a program's matrix in shared memory while it fits (N <= 170 / 169) and with blocked
// kernels above that, so long horizons batch like short ones.
//
// A batch lives across many solves. Maximize with initialization_mode = warm start continues every
// program from the iterate of the previous solve (cone states, including the dual-recovery update,
// and the b / c scalings), with the NewtonControl warm-start logic of a single program: the warm centering
// schedule, and a restart from the identity for a program whose first factorisation fails or whose
// first step is too large (warmstart_abort_threshold). UpdateConstraintData replaces columns of a
// constraint's data in every program on the device, so that the next instance of a parametric
// problem is solved without building a new batch.
//
// Cones on variable subsets: each runs the cone kernels on its own m_k variables. Before each slack
// pass one gather copies their slices of y behind each program's y (the cone descriptors' y_offset
// points there); their Schur blocks go to scratch, and one scatter-add puts them into H, AW, AQc and
// the scalars after the full cones' kernels (the order of DenseKKTSolver::Assemble).
//
// Packed copies of the LMI operators: an update refreshes the lower triangles of the changed
// matrices only; data that is not symmetric bit for bit drops the cone's packed copy for the life of
// the batch (the slack passes then read the full matrices), as the constructor does.
#pragma once
#include <memory>
#include <vector>

#include "cone_program.h"

namespace conex {

struct BatchResult : ConexStatus {
  double by = 0, cx = 0, inv_sqrt_mu = 0;
  double b_scaling = 1, c_scaling = 1, d_inf = 0;
};

class BatchProgram {
 public:
  // All programs must have the same number of variables and the same list of constraints: cones
  // (LP, second-order, dense LMI; type, order, list of distinct variables — all of them in order, or
  // any subset in any order) and equality blocks (rows, variable subset) at the same positions among
  // them; at least one cone. Throws otherwise.
  explicit BatchProgram(const std::vector<Program*>& programs);
  ~BatchProgram();

  int size() const { return batch_; }
  int number_of_variables() const { return m_; }
  // b, y: m x B column-major host arrays. Returns the number of solved programs. A warm start
  // (config.initialization_mode != cold start) throws when the batch has never been solved.
  int Maximize(const double* b, const SolverConfiguration& config, double* y);
  // Replaces columns [first, first + count) of the data of constraint `constraint` (numbered like
  // GetDualVariable) in every program: cones [A | c] (rows x (m_k + 1) for a cone on m_k variables,
  // column j for its j-th variable; LMI: vec(A_j) and vec(C)),
  // equality blocks [A | b] (rows x (nvars + 1)). data: B host blocks of rows x count, column-major,
  // program p at data + p * rows * count. Throws on bad arguments before anything is written.
  void UpdateConstraintData(int constraint, int first, int count, const double* data);
  // The rows and columns of that data for `constraint`; false when there is no such constraint.
  bool ConstraintDataShape(int constraint, int* rows, int* columns) const;
  const std::vector<BatchResult>& results() const { return results_; }
  // Device milliseconds of the last Maximize (CUDA events on the batch's stream) and of its
  // individual Newton steps.
  double milliseconds() const { return total_ms_; }
  const std::vector<float>& step_milliseconds() const { return step_ms_; }
  // Scaling point of constraint `cone` of program `p`, rescaled like Program::GetDualVariable; the
  // numbering counts equality blocks, which have no dual variable (size 0, nothing written).
  int DualVariableSize(int cone) const;
  void GetDualVariable(int p, int cone, double* host_out);

 private:
  struct Impl;
  std::unique_ptr<Impl> impl_;
  int batch_ = 0, m_ = 0;
  std::vector<BatchResult> results_;
  std::vector<float> step_ms_;
  double total_ms_ = 0;
};

}  // namespace conex

// The conex C ABI (include/conex.h) on top of the device-resident Program — counterpart of the
// reference's interfaces/conex.cc. Dense/sparse LMI, LP, second-order-cone and equality constraints
// are device cones; the entry points that build cones outside the scope (Hermitian LMIs, quadratic
// costs) validate their arguments like the reference and then report failure on stderr instead of
// silently doing CPU work. Exceptions never cross the ABI: they map to the call's failure value.
#include <atomic>
#include <cuda_runtime_api.h>

#include <cstdlib>
#include <cstring>
#include <iostream>
#include <vector>

#include "../../../include/conex_b200.h"
#include "communicator.h"
#include "cone_program.h"
#include "dense_lmi_constraint.h"
#include "small_cone_constraint.h"
#include "supernodal_kkt_solver.h"
#include "batch_program.h"
#include <cmath>
#include "divergence.h"
#include "tridiagonal_eigenvalues.h"

namespace cxb {
std::atomic<long> g_launch_count{0};
}

using conex::DenseLMIConstraint;
using conex::EqualityConstraints;
using conex::LinearConstraint;
using conex::SOCConstraint;
using conex::Program;
using conex::SolverConfiguration;

namespace {

// reference interfaces/conex.cc:20-33 (SAFER_CAST_TO_Program): null check only; the reference's
// workspace-count heuristic has no device-side equivalent.
#define CAST_PROGRAM_OR_FAIL(x, prog)                  \
  CONEX_DEMAND(x, "Program pointer is null.");         \
  Program* prog = static_cast<Program*>(x);

SolverConfiguration Convert(const CONEX_SolverConfiguration* c) {
  // reference interfaces/conex.cc:65-90
  SolverConfiguration o;
  o.prepare_dual_variables = c->prepare_dual_variables;
  o.initialization_mode = c->initialization_mode;
  o.inv_sqrt_mu_max = c->inv_sqrt_mu_max;
  o.minimum_mu = c->minimum_mu;
  o.maximum_mu = c->maximum_mu;
  o.divergence_upper_bound = c->divergence_upper_bound;
  o.enable_line_search = c->enable_line_search;
  o.dinf_upper_bound = c->dinf_upper_bound;
  o.final_centering_steps = c->final_centering_steps;
  o.final_centering_tolerance = c->final_centering_tolerance;
  o.initial_centering_steps_warmstart = c->initial_centering_steps_warmstart;
  o.initial_centering_steps_coldstart = c->initial_centering_steps_coldstart;
  o.warmstart_abort_threshold = c->warmstart_abort_threshold;
  o.max_iterations = c->max_iterations;
  o.iterative_refinement_iterations = c->iterative_refinement_iterations;
  o.infeasibility_threshold = c->infeasibility_threshold;
  o.kkt_error_tolerance = c->kkt_error_tolerance;
  o.enable_rescaling = c->enable_rescaling;
  o.kkt_solver = c->kkt_solver;
  return o;
}

template <typename F>
auto Guard(F&& f, decltype(f()) on_error) -> decltype(f()) {
  try {
    return f();
  } catch (const std::exception& e) {
    std::cerr << e.what() << std::endl;
    return on_error;
  }
}

int NotOnHotPath(const char* what) {
  std::cerr << "conex-b200: " << what
            << " is outside the device hot path of this build (dense LMI / PSD cones only)."
            << std::endl;
  return CONEX_FAILURE;
}

}  // namespace

extern "C" {

void* CONEX_CreateConeProgram() {
  return Guard(
      []() -> void* {
        Program* p = new Program(0);
        const char* v = std::getenv("CONEX_VERBOSE");
        p->verbose = v && std::atoi(v) != 0;
        return p;
      },
      nullptr);
}

void CONEX_DeleteConeProgram(void* prog) { delete static_cast<Program*>(prog); }

CONEX_STATUS CONEX_SetNumberOfVariables(void* p, int m) {
  // reference interfaces/conex.cc:399-407
  CONEX_DEMAND(m >= 1, "Number of variables must be > 0.");
  CAST_PROGRAM_OR_FAIL(p, prg);
  CONEX_DEMAND(prg->GetNumberOfVariables() == 0, "Number of variables already set.");
  prg->SetNumberOfVariables(m);
  return CONEX_SUCCESS;
}

int CONEX_AddDenseLMIConstraint(void* prog, const double* A, int Ar, int Ac, int m, const double* c,
                                int cr, int cc) {
  // reference interfaces/conex.cc:137-160. A program created without SetNumberOfVariables takes
  // its variable count from the first constraint.
  (void)Ac;
  (void)cr;
  (void)cc;
  return Guard(
      [&]() -> int {
        Program& program = *static_cast<Program*>(prog);
        if (program.GetNumberOfVariables() == 0) program.SetNumberOfVariables(m);
        const int id = program.NumberOfConstraints();
        if (program.AddConstraint(DenseLMIConstraint(Ar, m, A, c))) return -1;
        return id;
      },
      -1);
}

int CONEX_AddSparseLMIConstraint(void* prog, const double* A, int Ar, int Ac, int num_vars,
                                 const double* c, int cr, int cc, const long* vars, int vars_rows) {
  // reference interfaces/conex.cc:162-188
  (void)Ac;
  (void)cr;
  (void)cc;
  (void)vars_rows;
  return Guard(
      [&]() -> int {
        Program& program = *static_cast<Program*>(prog);
        std::vector<int> variables(num_vars);
        for (int i = 0; i < num_vars; i++) variables[i] = static_cast<int>(vars[i]);
        const int id = program.NumberOfConstraints();
        // duplicate or out-of-range variables: nothing was added, so `id` would name a later constraint
        if (program.AddConstraint(DenseLMIConstraint(Ar, num_vars, A, c), variables)) return -1;
        return id;
      },
      -1);
}

int CONEXB200_AddDenseLMIConstraintDevice(void* prog, const double* d_A, int n, int m,
                                          const double* d_C) {
  return Guard(
      [&]() -> int {
        Program& program = *static_cast<Program*>(prog);
        if (program.GetNumberOfVariables() == 0) program.SetNumberOfVariables(m);
        const int id = program.NumberOfConstraints();
        if (program.AddConstraint(DenseLMIConstraint(n, m, DenseLMIConstraint::DevicePointers{d_A, d_C}))) return -1;
        return id;
      },
      -1);
}

int CONEXB200_AddDenseLMIConstraintShard(void* prog, const double* d_A_local, int n, int m,
                                         const double* d_C) {
  return Guard(
      [&]() -> int {
        Program& program = *static_cast<Program*>(prog);
        if (program.GetNumberOfVariables() == 0) program.SetNumberOfVariables(m);
        const int id = program.NumberOfConstraints();
        program.AddConstraint(DenseLMIConstraint(n, m, DenseLMIConstraint::Sharded{},
                                                 DenseLMIConstraint::DevicePointers{d_A_local, d_C}));
        program.ctx_.collective = conex::Communicator::Get().distributed();
        return id;
      },
      -1);
}

int CONEXB200_NewDenseLMIConstraintStorage(void* prog, int n, int m, double** d_A_local, double** d_C) {
  return Guard(
      [&]() -> int {
        Program& program = *static_cast<Program*>(prog);
        if (program.GetNumberOfVariables() == 0) program.SetNumberOfVariables(m);
        const int id = program.NumberOfConstraints();
        DenseLMIConstraint cone(n, m, DenseLMIConstraint::Sharded{}, DenseLMIConstraint::Uninitialized{});
        // copies of the cone share one Storage (shared_ptr), so these pointers stay valid
        *d_A_local = cone.mutable_device_matrices();
        *d_C = cone.mutable_device_matrices() + static_cast<size_t>(n) * n * cone.local_matrices();
        program.AddConstraint(cone);
        program.ctx_.collective = conex::Communicator::Get().distributed();
        return id;
      },
      -1);
}

int CONEXB200_CommGetUniqueId(char* out128) {
  return Guard(
      [&]() -> int {
        conex::Communicator::Get().GetUniqueId(out128);
        return 0;
      },
      1);
}

int CONEXB200_CommInitRank(int world, int rank, const char* id128) {
  return Guard(
      [&]() -> int {
        conex::Communicator::Get().InitRank(world, rank, id128);
        return 0;
      },
      1);
}

void CONEXB200_CommDestroy(void) { conex::Communicator::Get().Destroy(); }
int CONEXB200_CommWorld(void) { return conex::Communicator::Get().world(); }
int CONEXB200_CommRank(void) { return conex::Communicator::Get().rank(); }

void CONEXB200_ShardRange(int m, int world, int rank, int* begin, int* count) {
  *begin = conex::ShardBegin(m, world, rank);
  *count = conex::ShardBegin(m, world, rank + 1) - *begin;
}

int CONEXB200_ShardPlan(int m, int world, int rank, int* out5, int capacity) {
  const auto plan = conex::ShardPlan(m, world, rank);
  int k = 0;
  for (const auto& t : plan) {
    if (k < capacity) {
      const int v[5] = {t.peer, t.row_begin, t.row_count, t.col_begin, t.col_count};
      std::memcpy(out5 + 5 * k, v, sizeof(v));
    }
    k++;
  }
  return k;
}

void CONEXB200_SetKKTSolverKind(void* prog, int kind) {
  if (prog && kind >= 0 && kind <= 2) static_cast<Program*>(prog)->kkt_solver_kind = kind;
}

int CONEXB200_GetNumberOfSupernodes(void* prog) {
  if (!prog) return -1;
  Program& program = *static_cast<Program*>(prog);
  return program.solver ? program.solver->NumberOfSupernodes() : 0;
}

int CONEXB200_SupernodalAnalysis(int N, int num_cliques, const int* clique_ptr, const int* clique_vars,
                                 int* position, int* node_of, int* node_ptr, int* node_vars, int* sep_ptr,
                                 int* sep_vars, int sep_capacity, double* flops2) {
  return Guard(
      [&]() -> int {
        std::vector<std::vector<int>> cliques(num_cliques);
        for (int c = 0; c < num_cliques; c++) {
          cliques[c].assign(clique_vars + clique_ptr[c], clique_vars + clique_ptr[c + 1]);
        }
        const conex::SupernodalStructure st = conex::AnalyzeCliques(N, cliques);
        const int nodes = static_cast<int>(st.supernodes.size());
        long seps = 0;
        for (const auto& s : st.separators) seps += static_cast<long>(s.size());
        if (seps > sep_capacity) return -static_cast<int>(std::min<long>(seps, 2000000000L));
        int a = 0, b = 0;
        for (int k = 0; k < nodes; k++) {
          node_ptr[k] = a;
          sep_ptr[k] = b;
          for (int v : st.supernodes[k]) node_vars[a++] = v;
          for (int v : st.separators[k]) sep_vars[b++] = v;
        }
        node_ptr[nodes] = a;
        sep_ptr[nodes] = b;
        for (int v = 0; v < N; v++) {
          position[v] = st.position[v];
          node_of[v] = st.node_of[v];
        }
        if (flops2) {
          flops2[0] = st.factor_flops;
          flops2[1] = st.dense_flops;
        }
        return nodes;
      },
      -1);
}

void CONEXB200_SetCollective(void* prog, int collective) {
  if (prog) static_cast<Program*>(prog)->ctx_.collective = collective != 0;
}

void CONEXB200_SetDistributedCholesky(int min_order, int block) {
  auto& policy = conex::DistributedCholeskyConfig();
  if (min_order >= 0) policy.min_order = min_order;
  if (block > 0) policy.block = block;
}

int CONEXB200_CholeskySchedule(int N, int block, int world, int rank, int* out3, int capacity) {
  const auto ops = conex::CholeskySchedule(N, block, world, rank);
  int k = 0;
  for (const auto& op : ops) {
    if (k < capacity) {
      const int v[3] = {op.kind, op.panel, op.target};
      std::memcpy(out3 + 3 * k, v, sizeof(v));
    }
    k++;
  }
  return k;
}

int CONEXB200_DistributedPotrf(int N, double* d_H, long ld, int block, int* info) {
  return Guard(
      [&]() -> int {
        conex::DeviceContext ctx;
        conex::DistributedCholesky chol;
        chol.Factor(ctx.cuda_stream(), N, d_H, ld, ctx.flags(), block);
        ctx.DownloadInts(info, ctx.flags(), 1);
        return 0;
      },
      1);
}

int CONEX_Maximize(void* prog_ptr, const double* b, int br, const CONEX_SolverConfiguration* config,
                   double* y, int yr) {
  // reference interfaces/conex.cc:93-105
  (void)yr;
  return Guard(
      [&]() -> int {
        Program& prog = *static_cast<Program*>(prog_ptr);
        std::vector<double> blinear(b, b + br);
        return conex::Solve(blinear, prog, Convert(config), y) ? 1 : 0;
      },
      0);
}

int CONEX_Solve(void* prog_ptr, const CONEX_SolverConfiguration* config, double* y, int yr) {
  // reference interfaces/conex.cc:107-112
  (void)yr;
  return Guard(
      [&]() -> int {
        Program& prog = *static_cast<Program*>(prog_ptr);
        return conex::Solve(prog, Convert(config), y) ? 1 : 0;
      },
      0);
}

void CONEX_GetDualVariable(void* prog_ptr, int i, double* x, int xr, int xc) {
  // reference interfaces/conex.cc:114-122
  // The reference only asserts size == xr * xc (compiled out under NDEBUG) and then writes `size` doubles
  // into the caller's buffer; a wrong shape is refused here instead of overrunning it.
  Guard(
      [&]() -> int {
        Program& prog = *static_cast<Program*>(prog_ptr);
        if (x == nullptr || i < 0 || i >= prog.NumberOfConstraints()) {
          std::cerr << "CONEX_GetDualVariable: invalid constraint or null buffer." << std::endl;
          return 0;
        }
        const long size = prog.GetDualVariableSize(i);
        if (static_cast<long>(xr) * xc != size) {
          std::cerr << "CONEX_GetDualVariable: buffer is " << xr << " x " << xc << " but the dual variable of constraint "
                    << i << " has " << size << " entries; nothing written." << std::endl;
          return 0;
        }
        prog.GetDualVariable(i, x);
        return 0;
      },
      0);
}

int CONEX_GetDualVariableSize(void* prog_ptr, int i) {
  return Guard([&]() -> int { return static_cast<Program*>(prog_ptr)->GetDualVariableSize(i); }, 1);
}

void CONEX_SetDefaultOptions(CONEX_SolverConfiguration* c) {
  // reference interfaces/conex.cc:231-257; additionally sets the two fields the reference forgets
  // (iterative_refinement_iterations, kkt_solver), which callers with stack structs otherwise
  // pass uninitialised.
  if (c == nullptr) {
    std::cerr << "Received null pointer.";
    return;
  }
  const SolverConfiguration d;
  c->prepare_dual_variables = d.prepare_dual_variables;
  c->initialization_mode = d.initialization_mode;
  c->inv_sqrt_mu_max = d.inv_sqrt_mu_max;
  c->minimum_mu = d.minimum_mu;
  c->maximum_mu = d.maximum_mu;
  c->divergence_upper_bound = d.divergence_upper_bound;
  c->enable_line_search = d.enable_line_search;
  c->dinf_upper_bound = d.dinf_upper_bound;
  c->final_centering_steps = d.final_centering_steps;
  c->final_centering_tolerance = d.final_centering_tolerance;
  c->initial_centering_steps_warmstart = d.initial_centering_steps_warmstart;
  c->initial_centering_steps_coldstart = d.initial_centering_steps_coldstart;
  c->warmstart_abort_threshold = d.warmstart_abort_threshold;
  c->max_iterations = d.max_iterations;
  c->iterative_refinement_iterations = d.iterative_refinement_iterations;
  c->infeasibility_threshold = d.infeasibility_threshold;
  c->kkt_error_tolerance = d.kkt_error_tolerance;
  c->enable_rescaling = d.enable_rescaling;
  c->kkt_solver = d.kkt_solver;
}

void CONEX_GetIterationStats(void* prog, CONEX_IterationStats* stats, int iter_num_circular) {
  // reference interfaces/conex.cc:259-285
  if (prog == nullptr || stats == nullptr) {
    std::cerr << "Received null pointer.";
    return;
  }
  Program& program = *static_cast<Program*>(prog);
  if (!program.stats.initialized) {
    std::cerr << "No statistics available.";
    return;
  }
  int iter = iter_num_circular;
  if (iter < 0) iter = program.stats.num_iter + iter;
  if (program.stats.num_iter <= iter || iter < 0) {
    std::cerr << "Specified iteration is out of bounds.";
    return;
  }
  const double k = program.stats.sqrt_inv_mu[iter];
  stats->mu = 1.0 / (k * k);
  stats->iteration_number = iter;
}

// ---- LP cone, second-order cone, equality constraints ------------------------------------------
int CONEX_AddDenseLinearConstraint(void* prog, const double* A, int Ar, int Ac, const double* c, int cr) {
  // reference interfaces/conex.cc:216-229: Ar rows, Ac variables, column-major A
  (void)cr;
  return Guard(
      [&]() -> int {
        Program& program = *static_cast<Program*>(prog);
        if (program.GetNumberOfVariables() == 0) program.SetNumberOfVariables(Ac);
        const int id = program.NumberOfConstraints();
        program.AddConstraint(LinearConstraint(Ar, Ac, A, c));
        return id;
      },
      -1);
}

int CONEX_AddLinearInequalities(void* prog, const double* A, int Ar, int Ac, const double* lb, int num_lb,
                                const double* ub, int num_ub) {
  // reference interfaces/conex.cc:190-215 + PreprocessLinearInequality (linear_constraint.cc:21-46):
  // rows with lb == ub become scaled equality constraints, finite bounds scaled inequality rows.
  (void)num_lb;
  (void)num_ub;
  return Guard(
      [&]() -> int {
        Program& program = *static_cast<Program*>(prog);
        std::vector<std::vector<double>> ineq_rows, eq_rows;
        std::vector<double> ineq_rhs, eq_rhs;
        for (int i = 0; i < Ar; i++) {
          double rr = 0;
          for (int j = 0; j < Ac; j++) rr += A[static_cast<size_t>(j) * Ar + i] * A[static_cast<size_t>(j) * Ar + i];
          auto row = [&](double scale) {
            std::vector<double> r(Ac);
            for (int j = 0; j < Ac; j++) r[j] = scale * A[static_cast<size_t>(j) * Ar + i];
            return r;
          };
          if (lb[i] == ub[i]) {
            const double scale = 1.0 / std::sqrt(rr + ub[i] * ub[i]);
            eq_rows.push_back(row(scale));
            eq_rhs.push_back(scale * ub[i]);
          } else {
            if (ub[i] < 1e8) {
              const double scale = 1.0 / std::sqrt(rr + ub[i] * ub[i]);
              ineq_rows.push_back(row(scale));
              ineq_rhs.push_back(scale * ub[i]);
            }
            if (lb[i] > -1e8) {
              const double scale = 1.0 / std::sqrt(rr + lb[i] * lb[i]);
              ineq_rows.push_back(row(-scale));
              ineq_rhs.push_back(-scale * lb[i]);
            }
          }
        }
        auto pack = [&](const std::vector<std::vector<double>>& rows) {
          const size_t r = rows.size();
          std::vector<double> M(r * Ac);
          for (size_t i = 0; i < r; i++)
            for (int j = 0; j < Ac; j++) M[static_cast<size_t>(j) * r + i] = rows[i][j];
          return M;
        };
        if (!ineq_rows.empty()) {
          const auto M = pack(ineq_rows);
          program.AddConstraint(LinearConstraint(static_cast<int>(ineq_rows.size()), Ac, M.data(), ineq_rhs.data()));
        }
        if (!eq_rows.empty()) {
          const auto M = pack(eq_rows);
          program.AddConstraint(EqualityConstraints(static_cast<int>(eq_rows.size()), Ac, M.data(), eq_rhs.data()));
        }
        return -1;  // the reference never returns an id here (conex.cc:213-214)
      },
      -1);
}

CONEX_STATUS CONEX_NewLorentzConeConstraint(void* p, int order, int* constraint_id) {
  // reference interfaces/conex.cc:384-397
  CONEX_DEMAND(order >= 1, "Received invalid n. Second order cone must have order (n + 1) >= 2.");
  CONEX_DEMAND(constraint_id, "Received output null pointer.");
  CAST_PROGRAM_OR_FAIL(p, prg);
  CONEX_DEMAND(prg->GetNumberOfVariables() >= 1, "Number of variables must be set first.");
  return Guard(
      [&]() -> int {
        prg->AddConstraint(SOCConstraint(order, prg->GetNumberOfVariables(), nullptr, nullptr));
        *constraint_id = prg->NumberOfConstraints() - 1;
        return CONEX_SUCCESS;
      },
      CONEX_FAILURE);
}

CONEX_STATUS CONEX_NewLinearInequality(void* p, int num_rows, int* constraint_id) {
  // reference interfaces/conex.cc:318-329
  CONEX_DEMAND(constraint_id, "Received output null pointer.");
  CAST_PROGRAM_OR_FAIL(p, prg);
  CONEX_DEMAND(num_rows >= 1 && prg->GetNumberOfVariables() >= 1, "Invalid dimensions.");
  return Guard(
      [&]() -> int {
        const bool status = prg->AddConstraint(LinearConstraint(num_rows, prg->GetNumberOfVariables(), nullptr, nullptr));
        *constraint_id = prg->NumberOfConstraints() - 1;
        return status ? CONEX_FAILURE : CONEX_SUCCESS;
      },
      CONEX_FAILURE);
}

CONEX_STATUS CONEX_UpdateLinearOperator(void* p, int constraint, double value, int variable, int row,
                                        int col, int hyper_complex_dim) {
  // reference interfaces/conex.cc:365-373, cone_program.h:147-159
  CAST_PROGRAM_OR_FAIL(p, prg);
  CONEX_DEMAND(constraint >= 0 && constraint < prg->NumberOfConstraints(), "Invalid Constraint.");
  return Guard(
      [&]() -> int {
        return UpdateLinearOperator(prg->constraints_[constraint], value, variable, row, col, hyper_complex_dim)
                   ? CONEX_FAILURE
                   : CONEX_SUCCESS;
      },
      CONEX_FAILURE);
}

CONEX_STATUS CONEX_UpdateAffineTerm(void* p, int constraint, double value, int row, int col,
                                    int hyper_complex_dim) {
  // reference interfaces/conex.cc:375-382
  CAST_PROGRAM_OR_FAIL(p, prg);
  CONEX_DEMAND(constraint >= 0 && constraint < prg->NumberOfConstraints(), "Invalid Constraint.");
  return Guard(
      [&]() -> int {
        return UpdateAffineTerm(prg->constraints_[constraint], value, row, col, hyper_complex_dim) ? CONEX_FAILURE
                                                                                                  : CONEX_SUCCESS;
      },
      CONEX_FAILURE);
}

// C++-only constructors of the reference exposed for tests and the batched bench:
// SOCConstraint(A, c) (soc_constraint.h:9-15); A is (n + 1) x m column-major.
int CONEXB200_AddSocConstraint(void* prog, int n, int m, const double* A, const double* c) {
  return Guard(
      [&]() -> int {
        Program& program = *static_cast<Program*>(prog);
        if (program.GetNumberOfVariables() == 0) program.SetNumberOfVariables(m);
        const int id = program.NumberOfConstraints();
        program.AddConstraint(SOCConstraint(n, m, A, c));
        return id;
      },
      -1);
}

// The LP cone and the second-order cone on a list of variables, like CONEX_AddSparseLMIConstraint for LMIs:
// c - A y[vars] >= 0 (A is rows x nvars) and c - A y[vars] in the Lorentz cone of order n + 1 (A is (n + 1) x nvars),
// column-major. Duplicate or out-of-range variables add nothing and return -1; otherwise the constraint id.
int CONEXB200_AddSparseLinearConstraint(void* prog, const double* A, int rows, int nvars, const double* c,
                                        const long* vars) {
  return Guard(
      [&]() -> int {
        Program& program = *static_cast<Program*>(prog);
        if (rows < 1 || nvars < 1 || !vars) return -1;
        std::vector<int> variables(nvars);
        for (int i = 0; i < nvars; i++) variables[i] = static_cast<int>(vars[i]);
        const int id = program.NumberOfConstraints();
        if (program.AddConstraint(LinearConstraint(rows, nvars, A, c), variables)) return -1;
        return id;
      },
      -1);
}

int CONEXB200_AddSparseSocConstraint(void* prog, int n, int nvars, const double* A, const double* c,
                                     const long* vars) {
  return Guard(
      [&]() -> int {
        Program& program = *static_cast<Program*>(prog);
        if (n < 1 || nvars < 1 || !vars) return -1;
        std::vector<int> variables(nvars);
        for (int i = 0; i < nvars; i++) variables[i] = static_cast<int>(vars[i]);
        const int id = program.NumberOfConstraints();
        if (program.AddConstraint(SOCConstraint(n, nvars, A, c), variables)) return -1;
        return id;
      },
      -1);
}

// Program::AddConstraint(EqualityConstraints{A, b}[, vars]) (cone_program.h:193-217); A is
// rows x nvars column-major, vars == NULL: all variables. Returns the constraint id or -1.
int CONEXB200_AddEqualityConstraint(void* prog, int rows, int nvars, const double* A, const double* b,
                                    const long* vars) {
  return Guard(
      [&]() -> int {
        Program& program = *static_cast<Program*>(prog);
        const int id = program.NumberOfConstraints();
        bool failed;
        if (vars) {
          std::vector<int> v(nvars);
          for (int i = 0; i < nvars; i++) v[i] = static_cast<int>(vars[i]);
          failed = program.AddConstraint(EqualityConstraints(rows, nvars, A, b), v);
        } else {
          failed = program.AddConstraint(EqualityConstraints(rows, nvars, A, b));
        }
        return failed ? -1 : id;
      },
      -1);
}

// ---- batched solves of structurally identical programs (batch_program.h) --------------------------
void* CONEXB200_CreateBatch(void* const* programs, int count) {
  return Guard(
      [&]() -> void* {
        std::vector<Program*> v(count);
        for (int i = 0; i < count; i++) v[i] = static_cast<Program*>(programs[i]);
        return new conex::BatchProgram(v);
      },
      nullptr);
}

void CONEXB200_DeleteBatch(void* batch) { delete static_cast<conex::BatchProgram*>(batch); }

int CONEXB200_BatchMaximize(void* batch, const double* b, const CONEX_SolverConfiguration* config, double* y,
                            int* solved) {
  return Guard(
      [&]() -> int {
        auto* bp = static_cast<conex::BatchProgram*>(batch);
        const int n = bp->Maximize(b, Convert(config), y);
        if (solved) {
          for (int p = 0; p < bp->size(); p++) solved[p] = bp->results()[p].solved;
        }
        return n;
      },
      -1);
}

void CONEXB200_BatchGetResults(void* batch, int* iterations, double* by, double* cx, double* inv_sqrt_mu) {
  auto* bp = static_cast<conex::BatchProgram*>(batch);
  for (int p = 0; p < bp->size(); p++) {
    const auto& r = bp->results()[p];
    if (iterations) iterations[p] = r.num_iterations;
    if (by) by[p] = r.by;
    if (cx) cx[p] = r.cx;
    if (inv_sqrt_mu) inv_sqrt_mu[p] = r.inv_sqrt_mu;
  }
}

double CONEXB200_BatchMilliseconds(void* batch) { return static_cast<conex::BatchProgram*>(batch)->milliseconds(); }

int CONEXB200_BatchStepMilliseconds(void* batch, double* out, int capacity) {
  const auto& v = static_cast<conex::BatchProgram*>(batch)->step_milliseconds();
  for (int i = 0; i < static_cast<int>(v.size()) && i < capacity; i++) out[i] = v[i];
  return static_cast<int>(v.size());
}

int CONEXB200_BatchGetDualVariable(void* batch, int program, int cone, double* x) {
  return Guard(
      [&]() -> int {
        auto* bp = static_cast<conex::BatchProgram*>(batch);
        bp->GetDualVariable(program, cone, x);
        return bp->DualVariableSize(cone);
      },
      -1);
}

int CONEXB200_BatchUpdateConstraintData(void* batch, int constraint, int first, int count, const double* data) {
  return Guard(
      [&]() -> int {
        static_cast<conex::BatchProgram*>(batch)->UpdateConstraintData(constraint, first, count, data);
        return 0;
      },
      -1);
}

int CONEXB200_BatchConstraintDataShape(void* batch, int constraint, int* rows, int* columns) {
  int r = 0, c = 0;
  if (!static_cast<conex::BatchProgram*>(batch)->ConstraintDataShape(constraint, &r, &c)) return -1;
  if (rows) *rows = r;
  if (columns) *columns = c;
  return 0;
}

// 1 when constraint `id` is an incremental LMI currently held in entry-sparse form (after the first
// solve / assembly), 0 when dense, -1 for other constraint types.
int CONEXB200_ConstraintIsEntrySparse(void* prog, int id) {
  Program& program = *static_cast<Program*>(prog);
  int k = 0;
  for (auto& c : program.eqs) {
    if (k++ != id) continue;
    if (auto* h = std::any_cast<conex::HermitianPsdConstraint>(&c.obj)) return h->entry_sparse() ? 1 : 0;
    return -1;
  }
  return -1;
}

int CONEXB200_GetAssemblyForm(void* prog, int id) {
  Program& program = *static_cast<Program*>(prog);
  int k = 0;
  for (auto& c : program.eqs) {
    if (k++ != id) continue;
    if (auto* h = std::any_cast<conex::HermitianPsdConstraint>(&c.obj)) return h->assembly_form();
    if (auto* d = std::any_cast<conex::DenseLMIConstraint>(&c.obj)) return d->assembly_form();
    return -1;
  }
  return -1;
}

void CONEXB200_SetPeerMemoryExchange(void* prog, int enabled) {
  static_cast<Program*>(prog)->ctx_.peer_memory_exchange = enabled != 0;
}

int CONEXB200_GetShardPhaseMilliseconds(void* prog, int id, double* out4) {
  Program& program = *static_cast<Program*>(prog);
  int k = 0;
  for (auto& c : program.eqs) {
    if (k++ != id) continue;
    if (auto* d = std::any_cast<conex::DenseLMIConstraint>(&c.obj)) return d->shard_phase_milliseconds(out4) ? 1 : 0;
    return 0;
  }
  return 0;
}

int CONEXB200_SizeOfKKTSystem(void* prog) { return static_cast<Program*>(prog)->SizeOfKKTSystem(); }

// Host-logic probe: pivot order of the regularised LDL^T from the diagonal (RLDLT.h:328-356).
void CONEXB200_RldltPivotOrder(int n, const double* diag, int* perm) {
  const auto p = conex::RldltPivotOrderForTest(std::vector<double>(diag, diag + n));
  for (int i = 0; i < n; i++) perm[i] = p[i];
}

// ---- entry points whose cones are not on the device hot path ------------------------------------
int CONEX_AddQuadraticCost(void*, const double*, int, int) {
  return NotOnHotPath("CONEX_AddQuadraticCost");
}
CONEX_STATUS CONEX_NewLinearMatrixInequality(void* p, int order, int hyper_complex_dim,
                                             int* constraint_id) {
  // argument validation as in the reference (interfaces/conex.cc:287-316)
  CONEX_DEMAND(order >= 1, "Invalid LMI dimensions.");
  CONEX_DEMAND(constraint_id, "Received output null pointer.");
  CONEX_DEMAND(hyper_complex_dim == 1 || hyper_complex_dim == 2 || hyper_complex_dim == 4 ||
                   hyper_complex_dim == 8,
               "Hypercomplex dimension must be 1, 2, 4, or 8.");
  CAST_PROGRAM_OR_FAIL(p, prg);
  if (hyper_complex_dim != 1) {
    return NotOnHotPath("CONEX_NewLinearMatrixInequality over the complex / quaternion / octonion algebras");
  }
  CONEX_DEMAND(prg->GetNumberOfVariables() >= 1, "Number of variables must be set first.");
  return Guard(
      [&]() -> int {
        prg->AddConstraint(conex::HermitianPsdConstraint(order, prg->GetNumberOfVariables()));
        *constraint_id = prg->NumberOfConstraints() - 1;
        return CONEX_SUCCESS;
      },
      CONEX_FAILURE);
}
CONEX_STATUS CONEX_NewQuadraticCost(void* p, int* constraint_id) {
  CONEX_DEMAND(constraint_id, "Received output null pointer.");
  CONEX_DEMAND(p, "Program pointer is null.");
  return NotOnHotPath("CONEX_NewQuadraticCost");
}
CONEX_STATUS CONEX_UpdateQuadraticCostMatrix(void* p, int, double, int, int) {
  CONEX_DEMAND(p, "Program pointer is null.");
  return NotOnHotPath("CONEX_UpdateQuadraticCostMatrix");
}

// ---- CONEXB200_* extensions ----------------------------------------------------------------------
void CONEXB200_FeasibleObjective(void* prog, double* b) {
  Guard(
      [&]() -> int {
        const auto v = conex::GetFeasibleObjective(static_cast<Program*>(prog));
        std::memcpy(b, v.data(), sizeof(double) * v.size());
        return 0;
      },
      0);
}

void CONEXB200_GetStatus(void* prog, int* out4) {
  const conex::ConexStatus s = static_cast<Program*>(prog)->Status();
  out4[0] = s.solved;
  out4[1] = s.num_iterations;
  out4[2] = s.primal_infeasible;
  out4[3] = s.dual_infeasible;
}

int CONEXB200_GetIterationLog(void* prog, int iter, double* out8) {
  const auto& log = static_cast<Program*>(prog)->log;
  if (iter < 0 || iter >= static_cast<int>(log.size())) return 0;
  const auto& r = log[iter];
  const double v[8] = {r.inv_sqrt_mu, r.mu, r.d_2, r.d_inf, r.by, r.cx, r.kkt_error, r.step_size};
  std::memcpy(out8, v, sizeof(v));
  return 1;
}

int CONEXB200_GetObjectiveTerms(void* prog, int iter, double* out3) {
  const auto& log = static_cast<Program*>(prog)->log;
  if (iter < 0) iter += static_cast<int>(log.size());
  if (iter < 0 || iter >= static_cast<int>(log.size())) return 0;
  for (int p = 0; p < 3; p++) out3[p] = log[iter].cx_terms[p];
  return 1;
}

int CONEXB200_GetIterationMilliseconds(void* prog, int iter, double* ms) {
  const auto& log = static_cast<Program*>(prog)->log;
  if (iter < 0 || iter >= static_cast<int>(log.size())) return 0;
  *ms = log[iter].milliseconds;
  return 1;
}

int CONEXB200_GetIterationPhaseMilliseconds(void* prog, int iter, double* out5) {
  const auto& log = static_cast<Program*>(prog)->log;
  if (iter < 0 || iter >= static_cast<int>(log.size())) return 0;
  for (int p = 0; p < 5; p++) out5[p] = log[iter].phase_ms[p];
  return 1;
}

void CONEXB200_SetTiming(void* prog, int enabled) {
  static_cast<Program*>(prog)->timing_enabled = enabled != 0;
}

void CONEXB200_SetAssemblyMode(void* prog, int mode) {
  static_cast<Program*>(prog)->ctx_.assembly_mode = mode;
}

void CONEXB200_GetPhaseSeconds(void* prog, double* out5) {
  const auto& s = static_cast<Program*>(prog)->seconds;
  out5[0] = s.assemble;
  out5[1] = s.factor;
  out5[2] = s.solve;
  out5[3] = s.update;
  out5[4] = s.mu;
}

void CONEXB200_AssembleNewtonSystem(void* prog_ptr, int coldstart, double* H, double* AW,
                                    double* AQc, double* scalars2) {
  Guard(
      [&]() -> int {
        Program& prog = *static_cast<Program*>(prog_ptr);
        SolverConfiguration cfg;
        cfg.initialization_mode = coldstart ? conex::CONEX_INITIALIZATION_MODE_COLDSTART
                                            : conex::CONEX_INITIALIZATION_MODE_WARMSTART;
        conex::Initialize(prog, cfg);
        prog.solver->Assemble();
        // residual aggregation is internal to cone_program.cc; GetFeasibleObjective path reuses it
        const int m = prog.SizeOfKKTSystem();
        const conex::Ref Hd = prog.solver->KKTMatrix();
        if (cudaMemcpy2DAsync(H, sizeof(double) * m, Hd.data, sizeof(double) * Hd.ld,
                              sizeof(double) * m, m, cudaMemcpyDeviceToHost,
                              prog.ctx_.cuda_stream()) != cudaSuccess) {
          throw std::runtime_error("conex-b200: D2H copy of H failed");
        }
        prog.ctx_.Synchronize();
        conex::AssembleResidualsForExport(prog, AW, AQc, scalars2);
        return 0;
      },
      0);
}

// Host-logic probes (no GPU needed): the mu rule and the Jacobi-matrix eigenvalue extremes.
double CONEXB200_DivergenceUpperBoundInverse(double bound, double frobenius_norm_squared,
                                             double trace, double lambda_min, double lambda_max,
                                             double rank) {
  conex::WeightedSlackEigenvalues p;
  p.frobenius_norm_squared = frobenius_norm_squared;
  p.trace = trace;
  p.lambda_min = lambda_min;
  p.lambda_max = lambda_max;
  p.rank = rank;
  return conex::DivergenceUpperBoundInverse(bound, p);
}

void CONEXB200_TridiagonalExtremes(int n, const double* alpha, const double* beta, double* out2) {
  const auto mm = conex::ExtremeEigenvaluesOfTridiagonal(
      std::vector<double>(alpha, alpha + n), std::vector<double>(beta, beta + (n > 0 ? n - 1 : 0)));
  out2[0] = mm.first;
  out2[1] = mm.second;
}

void* CONEXB200_CreateConeProgramOnMemoryOf(void* other) {
  // reference: Program prog2(m, &prog.memory_) (cone_program.h:106-109)
  if (other == nullptr) return nullptr;
  try {
    Program* o = static_cast<Program*>(other);
    return new Program(0, o->workspace_data_);
  } catch (const std::exception& e) {
    std::cerr << e.what() << std::endl;
    return nullptr;
  }
}

int CONEXB200_NumberOfConstraints(void* prog_ptr) {
  return Guard([&]() -> int { return static_cast<Program*>(prog_ptr)->NumberOfConstraints(); }, -1);
}

long CONEXB200_LaunchCount() { return cxb::g_launch_count.load(); }

int CONEXB200_DeviceAvailable() {
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return 0;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, 0) != cudaSuccess) return 0;
  return prop.major == 10 ? 1 : 0;
}

}  // extern "C"

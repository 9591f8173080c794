#include "cone_program.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <iomanip>
#include <limits>
#include <set>

#include "../../../include/conex_b200_device.h"
#include "communicator.h"
#include "newton_control.h"
#include "supernodal_kkt_solver.h"

namespace conex {

// ================================================================================================
// Dense KKT solver
// ================================================================================================

DenseKKTSolver::DenseKKTSolver(DeviceContext* ctx, int N)
    : ctx_(ctx), N_(N), ldh_(WorkspaceSchurComplement::AugLd(N)) {
  H_.Resize(static_cast<size_t>(ldh_) * (N + 2));
}

void DenseKKTSolver::Bind(std::list<Container>* eqs) {
  eqs_ = eqs;
  has_direct_ = false;
  for (auto& c : *eqs) {
    const int mc = static_cast<int>(c.variables.size());
    c.identity_clique = (mc == N_);
    for (int i = 0; i < mc && c.identity_clique; i++) c.identity_clique = (c.variables[i] == i);
    c.direct_update = c.identity_clique && !has_direct_;
    if (c.direct_update) has_direct_ = true;
    c.submatrix_data_.m_ = mc;
    c.submatrix_data_.residual_only_ = c.direct_update;  // its G aliases H
    if (!c.identity_clique) {
      c.d_variables.Resize(mc);
      // stream-ordered: the program's stream does not synchronise with the legacy default stream
      CudaCheck(cudaMemcpyAsync(c.d_variables.get(), c.variables.data(), sizeof(int) * mc,
                                cudaMemcpyHostToDevice, ctx_->cuda_stream()),
                "upload of clique indices");
      c.y_clique.Resize(mc);
    }
  }
}

void DenseKKTSolver::Assemble() {
  void* s = ctx_->stream();
  // The aliasing cone assigns every entry of the lower triangle, so it goes first
  // (reference: root clique processed first, kkt_solver.cc:164-170).
  for (auto& c : *eqs_) {
    if (!c.direct_update) continue;
    c.submatrix_data_.G = KKTMatrix();
    ConstructSchurComplementSystem(&c.constraint, true, &c.submatrix_data_);
  }
  if (!has_direct_) ctx_->Zero(H_.get(), H_.size());
  for (auto& c : *eqs_) {
    if (c.direct_update) continue;
    ConstructSchurComplementSystem(&c.constraint, true, &c.submatrix_data_);
    const int mc = c.submatrix_data_.m_;
    if (c.identity_clique) {
      // same index set as H: add the lower triangle column by column through the scatter kernel
      // with an identity map
      if (c.d_variables.size() == 0) {
        std::vector<int> id(mc);
        for (int i = 0; i < mc; i++) id[i] = i;
        c.d_variables.Resize(mc);
        CudaCheck(cudaMemcpyAsync(c.d_variables.get(), id.data(), sizeof(int) * mc, cudaMemcpyHostToDevice,
                                  ctx_->cuda_stream()),
                  "upload of clique indices");
        ctx_->Synchronize();  // `id` is a local
      }
    }
    DeviceCheck(cxb_scatter_add_lower(s, mc, c.submatrix_data_.G.data, c.submatrix_data_.G.ld,
                                      c.d_variables.get(), H_.get(), ldh_),
                "cxb_scatter_add_lower");
  }
}

namespace {

// The pivot order of Eigen::RLDLT (RLDLT.h:328-356): at step k the largest |diagonal entry| among
// positions k.. of the *current* arrangement (first occurrence on ties) is swapped to position k.
// The left-looking algorithm has not touched those entries yet, so they are the original diagonal
// and the whole order follows from it. Returns perm with perm[k] = original index at position k.
std::vector<int> RldltPivotOrder(const std::vector<double>& diag) {
  const int n = static_cast<int>(diag.size());
  std::vector<int> at(n);  // position -> original index
  for (int i = 0; i < n; i++) at[i] = i;
  // candidates ordered by (-|d|, position)
  std::set<std::pair<double, int>> pool;
  for (int i = 0; i < n; i++) pool.insert({-std::fabs(diag[i]), i});
  for (int k = 0; k < n; k++) {
    const auto best = *pool.begin();
    const int p = best.second;
    pool.erase(pool.begin());
    if (p != k) {
      // the element at position k moves to position p and stays a candidate
      pool.erase({-std::fabs(diag[at[k]]), k});
      std::swap(at[k], at[p]);
      pool.insert({-std::fabs(diag[at[p]]), p});
    }
  }
  return at;
}

}  // namespace

std::vector<int> RldltPivotOrderForTest(const std::vector<double>& diag) { return RldltPivotOrder(diag); }

void DenseKKTSolver::FactorLDLT() {
  // reference block_triangular_operations.cc:315-349 + RLDLT.h:297-431 for one dense supernode
  void* s = ctx_->stream();
  const int N = N_;
  if (Hp_.size() == 0) {
    Hp_.Resize(static_cast<size_t>(ldh_) * N);
    signs_.Resize(N);
    diag_.Resize(2 * static_cast<size_t>(N));
    ldlt_work_.Resize(cxb_ldlt_worksize(N));
    perm_.Resize(N);
  }
  DeviceCheck(cxb_copy_strided(s, N, H_.get(), ldh_ + 1, diag_.get(), 1), "cxb_copy_strided");
  std::vector<double> d(N);
  ctx_->Download(d.data(), diag_.get(), N);
  host_perm_ = RldltPivotOrder(d);
  CudaCheck(cudaMemcpyAsync(perm_.get(), host_perm_.data(), sizeof(int) * N, cudaMemcpyHostToDevice,
                            ctx_->cuda_stream()),
            "upload of the pivot order");
  DeviceCheck(cxb_sym_permute_lower(s, N, H_.get(), ldh_, perm_.get(), Hp_.get(), ldh_), "cxb_sym_permute_lower");
  DeviceCheck(cxb_ldlt_lower(s, N, Hp_.get(), ldh_, signs_.get(), ldlt_work_.get(), ctx_->flags() + 2),
              "cxb_ldlt_lower");
  ctx_->Synchronize();  // host_perm_ is pageable
}

bool DenseKKTSolver::Factor() {
  if (mode_ == CONEX_QR_FACTORIZATION) {
    throw std::runtime_error("conex-b200: the QR KKT mode is not implemented on the device");
  }
  if (iterative_refinement_iterations_ > 0) {
    // keep the assembled matrix for the residuals (kkt_solver.cc:174-178)
    kkt_matrix_.Reserve(static_cast<size_t>(ldh_) * N_);
    ctx_->CopyOnDevice(kkt_matrix_.get(), H_.get(), static_cast<size_t>(ldh_) * N_);
  }
  if (num_dual_ > 0) {
    FactorLDLT();
    return true;  // the regularised LDL^T never fails (kkt_solver.cc:187-193)
  }
  int* info = ctx_->flags();
  const DistributedCholeskyPolicy& policy = DistributedCholeskyConfig();
  if (ctx_->collective && Communicator::Get().distributed() && N_ >= policy.min_order) {
    // H is replicated bit-identically (one all-reduce, or replicated deterministic kernels)
    distributed_.Factor(ctx_->cuda_stream(), N_, H_.get(), ldh_, info, policy.block);
  } else {
    DeviceCheck(cxb_potrf_lower(ctx_->stream(), N_, H_.get(), ldh_, nullptr, info), "cxb_potrf_lower");
  }
  int host_info = 0;
  ctx_->DownloadInts(&host_info, info, 1);
  return host_info == 0;  // reference block_triangular_operations.cc:193-196
}

void DenseKKTSolver::SolveOnce(double* rhs) const {
  if (num_dual_ > 0) {
    DeviceCheck(cxb_ldlt_solve(ctx_->stream(), N_, Hp_.get(), ldh_, signs_.get(), perm_.get(), rhs,
                               diag_.get() + N_),
                "cxb_ldlt_solve");
  } else {
    DeviceCheck(cxb_potrs_lower(ctx_->stream(), N_, H_.get(), ldh_, rhs, N_, 1), "cxb_potrs_lower");
  }
}

void DenseKKTSolver::SolveInPlace(Ref* b) const {
  // reference kkt_solver.cc:220-263
  void* s = ctx_->stream();
  for (int k = 0; k < b->cols; k++) {
    double* y = b->col(k);
    if (iterative_refinement_iterations_ <= 0) {
      SolveOnce(y);
      continue;
    }
    refine_.Reserve(3 * static_cast<size_t>(N_));
    double* total_residual = refine_.get();
    double* r = total_residual + N_;
    double* Ky = r + N_;
    ctx_->CopyOnDevice(total_residual, y, N_);
    SolveOnce(y);
    for (int it = 0; it < iterative_refinement_iterations_; it++) {
      DeviceCheck(cxb_symv_lower(s, N_, kkt_matrix_.get(), ldh_, y, Ky), "cxb_symv_lower");
      // r = total_residual - K y ; solve ; y += r
      DeviceCheck(cxb_axpbypcz(s, N_, 1.0, total_residual, 0.0, r, -1.0, Ky), "cxb_axpbypcz");
      SolveOnce(r);
      DeviceCheck(cxb_axpbypcz(s, N_, 1.0, r, 1.0, y, 0.0, nullptr), "cxb_axpbypcz");
    }
  }
}

// ================================================================================================
// Program
// ================================================================================================

bool Program::VariablesAreUnique(const std::vector<int>& x) const {
  std::vector<char> seen(num_variables_, 0);
  for (int v : x) {
    if (v < 0 || v >= num_variables_ || seen[v]) return false;
    seen[v] = 1;
  }
  return true;
}

bool Program::AddLinearCost(const std::vector<double>& b) {
  CONEX_DEMAND(static_cast<int>(b.size()) == GetNumberOfVariables(),
               "Cost vector dimension does not equal number of variables");
  for (size_t i = 0; i < b.size(); i++) linear_cost_[i] += b[i];
  return true;
}

void Program::InitializeWorkspace() {
  // Sizes first, then carve (reference workspace.h:27-35).
  size_t total = 0;
  for (auto& c : eqs) {
    Workspace w = c.constraint.workspace();
    total += WorkspaceSchurComplement::Aligned(SizeOf(w));
    total += SizeOf(c.submatrix_data_);
  }
  sys.m_ = SizeOfKKTSystem();
  sys.residual_only_ = true;
  total += SizeOf(sys);
  DeviceBuffer<double>& arena = workspace_data_->data;
  if (total > arena.size()) arena.Resize(total);  // only ever grows; a warm start keeps data
  double* p = arena.get();
  for (auto& c : eqs) {
    Workspace w = c.constraint.workspace();
    Initialize(&w, p);
    p += WorkspaceSchurComplement::Aligned(SizeOf(w));
    Initialize(&c.submatrix_data_, p);
    p += SizeOf(c.submatrix_data_);
  }
  Initialize(&sys, p);
  vectors_.Reserve(4 * WorkspaceSchurComplement::Aligned(sys.m_));
  is_initialized = true;
}

int Program::GetDualVariableSize(int i) {
  int cnt = 0;
  for (auto& c : eqs) {
    if (cnt++ == i) return c.constraint.dual_variable_size();
  }
  std::cerr << "Invalid Constraint" << std::endl;
  return 1;
}

void Program::GetDualVariable(int i, double* host_out) {
  int cnt = 0;
  for (auto& c : eqs) {
    if (cnt++ != i) continue;
    const Ref w = c.constraint.dual_variable();
    const size_t sz = w.size();
    ctx_.Download(host_out, w.data, sz);
    const double k = stats.num_iter > 0 ? stats.sqrt_inv_mu[stats.num_iter - 1] : 0;
    ScaleDualVariable(stats.num_iter, status_.primal_infeasible, k, stats.b_scaling, host_out, sz);
    return;
  }
}

bool Initialize(Program& prog, const SolverConfiguration& config) {
  // reference cone_program.cc:78-112
  if (prog.is_initialized && config.initialization_mode != CONEX_INITIALIZATION_MODE_COLDSTART) {
    return true;
  }
  prog.stats.initialized = true;
  // One dense supernode, or the multifrontal solver when the cones' cliques leave H block-sparse
  // (reference: SupernodalKKTSolver always; here the dense solver is the special case of one clique).
  const int N = prog.SizeOfKKTSystem();
  bool reused = false;
  std::unique_ptr<KKTSolver> fresh;
  // Iterative refinement needs K y with the assembled matrix (kkt_solver.cc:248-261); the multifrontal solver
  // factors its fronts in place and keeps no copy, so a configuration that asks for refinement gets the dense
  // solver unless the multifrontal one was requested explicitly (kind 2, which then fails loudly in SolveInPlace).
  const bool refinement_needs_dense = config.iterative_refinement_iterations > 0 && prog.kkt_solver_kind != 2;
  if (prog.kkt_solver_kind != 1 && !prog.ctx_.collective && !refinement_needs_dense) {
    std::vector<std::vector<int>> cliques;
    bool some_cone_couples_everything = false;
    for (const auto& c : prog.eqs) {
      cliques.push_back(c.variables);
      some_cone_couples_everything = some_cone_couples_everything || static_cast<int>(c.variables.size()) == N;
    }
    // Equality multipliers (indices >= number of variables) have a zero diagonal entry until the variables they couple
    // are eliminated; the LDL^T pivots only inside a supernode (like the reference's BlockLDLTInPlace), so a multiplier
    // eliminated before its variables would meet an exact zero pivot (regularised to 1e-9: a penalty method, 1e-8
    // residuals). For the symbolic step every clique that shares a variable with an equality block therefore also
    // carries that block's multipliers: a multiplier is then eliminated in a node at or above the nodes of all its
    // variables, and inside that node the pivot order by |diagonal| takes it after them.
    std::vector<std::vector<int>> analysis_cliques = cliques;
    {
      const int nv = prog.GetNumberOfVariables();
      for (size_t e = 0; e < cliques.size(); e++) {
        std::vector<int> multipliers;
        std::vector<char> touched(nv, 0);
        for (int v : cliques[e]) {
          if (v >= nv) multipliers.push_back(v); else touched[v] = 1;
        }
        if (multipliers.empty()) continue;
        for (size_t k = 0; k < cliques.size(); k++) {
          if (k == e) continue;
          bool shares = false;
          for (int v : cliques[k]) shares = shares || (v < nv && touched[v]);
          if (!shares) continue;
          for (int l : multipliers) {
            if (std::find(analysis_cliques[k].begin(), analysis_cliques[k].end(), l) == analysis_cliques[k].end()) {
              analysis_cliques[k].push_back(l);
            }
          }
        }
      }
    }
    // The symbolic step depends on the cliques alone: a repeated cold start of the same program keeps
    // the multifrontal solver with its destination lists (hundreds of ms of host work at order 10^4).
    if (prog.solver && prog.solver_is_multifrontal_ && prog.solver_order_ == N &&
        prog.solver_kind_ == prog.kkt_solver_kind && prog.solver_cliques_ == cliques) {
      reused = true;
    } else if (some_cone_couples_everything && prog.kkt_solver_kind != 2) {
      // one clique on all the variables (unique indices: VariablesAreUnique): a single dense supernode,
      // nothing to analyse
    } else {
      SupernodalStructure st = AnalyzeCliques(N, analysis_cliques);
      const bool pays = st.supernodes.size() > 1 && N >= 256 && st.factor_flops < 0.5 * st.dense_flops;
      if (prog.kkt_solver_kind == 2 || pays) {
        fresh = std::make_unique<SupernodalKKTSolver>(&prog.ctx_, N, std::move(st));
        prog.solver_cliques_ = std::move(cliques);
        prog.solver_order_ = N;
        prog.solver_kind_ = prog.kkt_solver_kind;
      }
    }
  } else if (prog.kkt_solver_kind == 2) {
    throw std::runtime_error("conex-b200: the supernodal KKT solver does not handle collective (multi-GPU) programs");
  }
  if (!reused) {
    prog.solver_is_multifrontal_ = fresh != nullptr;
    // the old solver's N x N buffers (3.2 GB each at m = 20000) are released before the new ones are allocated
    prog.solver.reset();
    if (!fresh) fresh = std::make_unique<DenseKKTSolver>(&prog.ctx_, N);
    prog.solver = std::move(fresh);
  }
  prog.solver->SetNumberOfMultipliers(prog.NumberOfMultipliers());
  if (!reused) prog.solver->Bind(&prog.eqs);
  prog.InitializeWorkspace();
  if (config.initialization_mode == CONEX_INITIALIZATION_MODE_COLDSTART) {
    prog.stats.b_scaling = 1;
    prog.stats.c_scaling = 1;
    for (auto* c : prog.constraints_) SetIdentity(c);
  }
  return true;
}

namespace {

// Aggregates the residual vectors of all cones (reference constraint_manager.h:107-124).
void AssembleSchurComplementResiduals(Program& prog) {
  void* s = prog.ctx_.stream();
  auto& sys = prog.sys;
  const int m = sys.m_;
  prog.ctx_.Zero(sys.AW, m);
  prog.ctx_.Zero(sys.AQc, m);
  prog.ctx_.Zero(sys.scalars, 2);
  for (auto& c : prog.eqs) {
    const auto& sub = c.submatrix_data_;
    const int* idx = c.identity_clique ? nullptr : c.d_variables.get();
    DeviceCheck(cxb_scatter_add_vec(s, sub.m_, sub.AW, idx, sys.AW), "cxb_scatter_add_vec");
    DeviceCheck(cxb_scatter_add_vec(s, sub.m_, sub.AQc, idx, sys.AQc), "cxb_scatter_add_vec");
    DeviceCheck(cxb_scatter_add_vec(s, 2, sub.scalars, nullptr, sys.scalars), "cxb_scatter_add_vec");
  }
}

// The clique's slice of y (reference cone_program.h:59-67 `Vars`).
Ref GatherVariables(Program& prog, Container& c, const Ref& y) {
  if (c.identity_clique) return y;
  const int mc = static_cast<int>(c.variables.size());
  DeviceCheck(cxb_gather_vec(prog.ctx_.stream(), mc, y.data, c.d_variables.get(), c.y_clique.get()),
              "cxb_gather_vec");
  return Ref(c.y_clique.get(), mc, 1);
}

// reference cone_program.h:69-90
void PrepareStep(Program& prog, const StepOptions& opt, const Ref& y, StepInfo* info) {
  info->normsqrd = 0;
  info->norminfd = -1;
  for (auto& c : prog.eqs) {
    StepInfo ci;
    PrepareStep(&c.constraint, opt, GatherVariables(prog, c, y), &ci);
    info->norminfd = std::max(info->norminfd, ci.norminfd);
    info->normsqrd += ci.normsqrd;
  }
}

// State of one solve besides its NewtonControl: the device vectors of the reference's Solve() locals
// (cone_program.cc:276-309).
class NewtonDriver {
 public:
  NewtonDriver(Program& prog, const SolverConfiguration& config)
      : prog_(prog), cfg_(config), ctx_(prog.ctx_), m_(prog.SizeOfKKTSystem()) {}

  bool Run(double* primal_variable);

 private:
  void UploadCost();
  WeightedSlackEigenvalues MuEigenvalues(const NewtonControl& ctl);
  void RecoverDualVariables(const NewtonControl& control);

  Program& prog_;
  const SolverConfiguration& cfg_;
  DeviceContext& ctx_;
  const int m_;
  double* d_b_ = nullptr;  // cost vector b (unscaled)
  double* d_y_ = nullptr;  // Newton direction / primal variable
  double* d_y2_ = nullptr;
  std::vector<double> b_;
};

void NewtonDriver::UploadCost() {
  const size_t stride = WorkspaceSchurComplement::Aligned(m_);
  d_b_ = prog_.vectors_.get();
  d_y_ = d_b_ + stride;
  d_y2_ = d_y_ + stride;
  b_.assign(m_, 0.0);  // zero cost on the multipliers (reference cone_program.cc:294-296)
  for (int i = 0; i < prog_.GetNumberOfVariables(); i++) b_[i] = -prog_.linear_cost_[i];
  CudaCheck(cudaMemcpyAsync(d_b_, b_.data(), sizeof(double) * m_, cudaMemcpyHostToDevice,
                            ctx_.cuda_stream()),
            "upload of b");
  ctx_.Synchronize();  // b_ is pageable: the copy must have consumed it before we move on
}

// The slack eigenvalues the mu rule reads (reference cone_program.cc:31-57, 173-191)
WeightedSlackEigenvalues NewtonDriver::MuEigenvalues(const NewtonControl& ctl) {
  // y = AQc*c_scaling - b*b_scaling ; y <- H^{-1} y
  DeviceCheck(cxb_axpbypcz(ctx_.stream(), m_, ctl.c_scaling(), prog_.sys.AQc, 0.0, d_y_, -ctl.b_scaling(), d_b_),
              "cxb_axpbypcz");
  Ref y(d_y_, m_, 1);
  static const bool trace = std::getenv("CONEX_TRACE_EIGEN") != nullptr;
  const auto t0 = std::chrono::high_resolution_clock::now();
  prog_.solver->SolveInPlace(&y);
  if (trace) {
    ctx_.Synchronize();
    std::cerr << "[conex-b200 trace] mu-phase solve (host wall, synchronised) "
              << std::chrono::duration<double, std::milli>(std::chrono::high_resolution_clock::now() - t0).count()
              << " ms" << std::endl;
  }
  SlackEigenvalueSum p;
  for (auto& c : prog_.eqs) {
    WeightedSlackEigenvalues t;
    GetWeightedSlackEigenvalues(&c.constraint, GatherVariables(prog_, c, y), ctl.c_scaling(), &t);
    p.Add(t.lambda_min, t.lambda_max, t.frobenius_norm_squared, t.trace);
  }
  return p;
}

// reference cone_program.cc:500-516
void NewtonDriver::RecoverDualVariables(const NewtonControl& control) {
  prog_.solver->Assemble();
  AssembleSchurComplementResiduals(prog_);
  prog_.solver->Factor();
  DeviceCheck(cxb_axpbypcz(ctx_.stream(), m_, control.k() * control.b_scaling(), d_b_, 0.0, d_y2_, -1.0, prog_.sys.AW),
              "cxb_axpbypcz");
  Ref y2(d_y2_, m_, 1);
  prog_.solver->SolveInPlace(&y2);
  StepOptions opt;
  opt.affine = true;
  opt.inv_sqrt_mu = control.k();
  opt.e_weight = 0;
  opt.c_weight = 0;
  StepInfo info;
  PrepareStep(prog_, opt, y2, &info);
}

bool NewtonDriver::Run(double* primal_variable) {
  auto& st = prog_.stats;
  auto& status = prog_.status_;
  status = ConexStatus();
  prog_.log.clear();
  prog_.seconds = PhaseSeconds();

  if (prog_.NumberOfConstraints() == 0) {
    // reference cone_program.cc:266-271
    for (int i = 0; i < prog_.GetNumberOfVariables(); i++) {
      primal_variable[i] = -prog_.linear_cost_[i] * std::numeric_limits<double>::infinity();
    }
    return false;
  }
  Initialize(prog_, cfg_);
  UploadCost();
  ctx_.Zero(d_y_, m_);
  st.sqrt_inv_mu.assign(std::max(cfg_.max_iterations, 1), 0.0);
  st.num_iter = 0;
  prog_.solver->SetIterativeRefinementIterations(cfg_.iterative_refinement_iterations);
  prog_.solver->SetSolverMode(cfg_.kkt_solver);

  int rank = 0;
  for (auto* c : prog_.constraints_) rank += Rank(*c);
  NewtonControl control(cfg_, rank, b_.data(), b_.size(), st.b_scaling, st.c_scaling);

  // Phase boundaries are CUDA events on the program stream: 0 start | 1 assembled | 2 factored |
  // 3 mu chosen | 4 solved | 5 updated (+ objective dots). Elapsed times are read after the
  // iteration's last synchronisation, so timing adds no host/device round trips.
  struct Events {
    cudaEvent_t e[6];
    Events() {
      for (auto& x : e) CudaCheck(cudaEventCreate(&x), "cudaEventCreate");
    }
    ~Events() {
      for (auto& x : e) cudaEventDestroy(x);
    }
  } ev;
  auto mark = [&](int i) { CudaCheck(cudaEventRecord(ev.e[i], ctx_.cuda_stream()), "cudaEventRecord"); };

  for (int i = 0; i < cfg_.max_iterations; i++) {
    if (!control.Begin(i)) break;
    mark(0);
    prog_.solver->Assemble();
    AssembleSchurComplementResiduals(prog_);
    mark(1);
    double aqc2 = 0;
    if (control.NeedsAqcNorm()) {
      DeviceCheck(cxb_dot(ctx_.stream(), m_, prog_.sys.AQc, prog_.sys.AQc, ctx_.scalars()), "cxb_dot");
      ctx_.Download(&aqc2, ctx_.scalars(), 1);
    }
    control.Rescale(aqc2);
    st.b_scaling = control.b_scaling();
    st.c_scaling = control.c_scaling();
    if (!prog_.solver->Factor()) {
      if (!control.RestartOnFactorizationFailure()) {
        status.solved = 0;
        return false;
      }
      for (auto* c : prog_.constraints_) SetIdentity(c);
      continue;
    }
    mark(2);
    if (control.update_mu() && cfg_.enable_line_search && !prog_.LineSearchAlwaysFails()) {
      // Programs made of LP cones only would run the reference's real line search, which is not built here.
      throw std::runtime_error("conex-b200: enable_line_search on LP-only programs is not implemented");
    }
    control.ChooseK(control.NeedsEigenvalues() ? MuEigenvalues(control) : WeightedSlackEigenvalues());
    const double k = control.k();
    mark(3);

    // y = k (b b_scaling + AQc c_scaling) - 2 AW   (reference cone_program.cc:409-411)
    DeviceCheck(cxb_axpbypcz(ctx_.stream(), m_, k * control.b_scaling(), d_b_, 0.0, d_y_, k * control.c_scaling(),
                             prog_.sys.AQc),
                "cxb_axpbypcz");
    DeviceCheck(cxb_axpbypcz(ctx_.stream(), m_, -2.0, prog_.sys.AW, 1.0, d_y_, 0.0, nullptr), "cxb_axpbypcz");
    Ref y(d_y_, m_, 1);
    prog_.solver->SolveInPlace(&y);
    mark(4);
    StepOptions opt;
    opt.affine = false;
    opt.inv_sqrt_mu = k;
    opt.e_weight = 1;
    opt.c_weight = k * control.c_scaling();
    StepInfo info;
    PrepareStep(prog_, opt, y, &info);
    if (control.Step(info.norminfd, info.normsqrd, &opt.step_size)) {
      for (auto* c : prog_.constraints_) TakeStep(c, opt);
    } else {
      for (auto* c : prog_.constraints_) SetIdentity(c);
    }
    // by, cx need b.y, AQc.y, <w,c>, <c,Qc>: one round trip of four doubles.
    DeviceCheck(cxb_dot(ctx_.stream(), m_, d_b_, d_y_, ctx_.scalars() + 0), "cxb_dot");
    DeviceCheck(cxb_dot(ctx_.stream(), m_, prog_.sys.AQc, d_y_, ctx_.scalars() + 1), "cxb_dot");
    ctx_.CopyOnDevice(ctx_.scalars() + 2, prog_.sys.scalars, 2);
    mark(5);
    double r[4];
    ctx_.Download(r, ctx_.scalars(), 4);
    float ms = 0;
    float phase_ms[5] = {0, 0, 0, 0, 0};
    cudaEventElapsedTime(&ms, ev.e[0], ev.e[5]);
    for (int p = 0; p < 5; p++) cudaEventElapsedTime(&phase_ms[p], ev.e[p], ev.e[p + 1]);
    prog_.seconds.assemble += 1e-3 * phase_ms[0];
    prog_.seconds.factor += 1e-3 * phase_ms[1];
    prog_.seconds.mu += 1e-3 * phase_ms[2];
    prog_.seconds.solve += 1e-3 * phase_ms[3];
    prog_.seconds.update += 1e-3 * phase_ms[4];

    const bool converged = control.End(r[0], r[1], r[2], r[3]);
    st.num_iter = control.num_iterations();
    st.sqrt_inv_mu[i] = k;
    prog_.log.push_back({k, control.mu(), control.d_2(), control.d_inf(), control.by(), control.cx(),
                         control.kkt_error(), opt.step_size, ms,
                         {phase_ms[0], phase_ms[1], phase_ms[2], phase_ms[3], phase_ms[4]},
                         {2 * r[2], r[1], k * r[3] * control.c_scaling()}});
    if (prog_.verbose) {
      std::cout << "i: " << std::setw(2) << i << ", mu: " << std::scientific << std::setprecision(2)
                << control.mu() << ", d_2: " << control.d_2() << ", d_inf: " << control.d_inf()
                << ", by: " << control.by() << ", cx: " << control.cx() << ", kkt_error: " << control.kkt_error()
                << ", ms: " << std::fixed << ms << std::endl;
    }
    if (converged) break;
  }

  ctx_.Download(primal_variable, d_y_, prog_.GetNumberOfVariables());  // yout = y.topRows(m), cone_program.cc:486
  if (cfg_.prepare_dual_variables) RecoverDualVariables(control);
  status = control.Finish(primal_variable, prog_.GetNumberOfVariables());
  ctx_.Synchronize();
  return status.solved != 0;
}

}  // namespace

bool Solve(Program& prog, const SolverConfiguration& config, double* primal_variable) {
  NewtonDriver driver(prog, config);
  return driver.Run(primal_variable);
}

bool Solve(const std::vector<double>& b, Program& prog, const SolverConfiguration& config,
           double* primal_variable) {
  prog.ClearLinearCosts();
  std::vector<double> minus_b(b.size());
  for (size_t i = 0; i < b.size(); i++) minus_b[i] = -b[i];
  prog.AddLinearCost(minus_b);
  return Solve(prog, config, primal_variable);
}

std::vector<double> GetFeasibleObjective(Program* prog) {
  Initialize(*prog, SolverConfiguration());
  prog->solver->Assemble();
  AssembleSchurComplementResiduals(*prog);
  const int m = prog->GetNumberOfVariables();
  std::vector<double> b(m);
  prog->ctx_.Download(b.data(), prog->sys.AW, m);
  for (auto& v : b) v *= .5;
  return b;
}

}  // namespace conex

namespace conex {
void AssembleResidualsForExport(Program& prog, double* AW, double* AQc, double* scalars2) {
  AssembleSchurComplementResiduals(prog);
  const int m = prog.SizeOfKKTSystem();
  prog.ctx_.Download(AW, prog.sys.AW, m);
  prog.ctx_.Download(AQc, prog.sys.AQc, m);
  prog.ctx_.Download(scalars2, prog.sys.scalars, 2);
}
}  // namespace conex

#include "batch_program.h"

#include <algorithm>
#include <cmath>
#include <cstring>

#include "../../../include/conex_b200_device.h"
#include "dense_lmi_constraint.h"
#include "equality_constraint.h"
#include "newton_control.h"
#include "small_cone_constraint.h"

namespace conex {

namespace {

struct ConeSlot {
  int type = 0, n = 0, m = 0, rows = 0;  // m: the number of the cone's variables
  std::vector<int> variables;            // empty for a cone on all variables in order (a full cone)
  size_t gather_offset = 0;              // subset cones: the slice of y (cxb_small_gather) ...
  size_t scratch_offset = 0;             // ... and the Schur block (cxb_small_scatter_schur) of each program
  size_t state_size = 0, work_size = 0;
  DeviceBuffer<double> data, state, work;
  DeviceBuffer<double> packed;  // LMI blocks: lower triangles of the matrices, for the slack passes
  cxb_small_cone desc;
  int rank = 0;
};

// An equality block A y[variables] = b: rank 0, no launches of its own. Its multipliers are the KKT unknowns
// m + offset .. m + offset + rows - 1; its rows of H, AQc and AW are constant and written once per batch.
struct EqualitySlot {
  int rows = 0, offset = 0;
  std::vector<int> variables;  // the columns of A
};

size_t Align4(size_t n) { return (n + 3) & ~static_cast<size_t>(3); }

}  // namespace

struct BatchProgram::Impl {
  DeviceContext ctx;
  std::vector<ConeSlot> cones;
  std::vector<cxb_small_cone> descs;  // the descriptors of `cones`, contiguous, for the fused launches
  std::vector<EqualitySlot> equalities;
  // constraint number -> index k into `cones`, or -1 - q for equalities[q]
  std::vector<int> slot_of;
  // N = m + multipliers: the order of the KKT systems (reference constraint_manager.h:42-48)
  int B = 0, m = 0, N = 0, multipliers = 0;
  long ldh = 0;
  size_t vstride = 0;
  // Cones on variable subsets (`subset`: their indices into `cones`, in constraint order). Each program's y and y2
  // carry the subset cones' slices of y behind the first vstride entries: ystride = vstride + gather_count. Their
  // Schur blocks are assigned into `sub_schur` (stride sub_stride per program) and scatter-added into H.
  std::vector<int> subset;
  int gather_count = 0;
  size_t ystride = 0, sub_stride = 0;
  DeviceBuffer<int> gather_idx, sub_table;
  DeviceBuffer<double> sub_schur;
  // per-program Newton system and vectors
  DeviceBuffer<double> H, AW, AQc, scal, b, y, y2;
  // with multipliers: the factors of the regularised LDL^T (H itself is kept, its equality rows are constant)
  DeviceBuffer<double> L, signs;
  DeviceBuffer<int> perm;
  // per-program scalars exchanged with the host each phase
  DeviceBuffer<double> coef;   // 3 x B coefficient arrays | B c_weights | B step sizes
  DeviceBuffer<double> out;    // cone outputs: B x ncones x 4, then B x 4 dots/scalars
  DeviceBuffer<int> info;      // B Cholesky flags | B Padé flags (| B regularisation flags of the LDL^T)
  DeviceBuffer<int> mask;      // B active | B mu-update | B aborted warm start
  DeviceBuffer<int> asymmetric;  // UpdateConstraintData: set when new LMI data is not symmetric
  PinnedBuffer<double> hcoef, hout;
  PinnedBuffer<int> hinfo, hmask;
  int rank = 0;
  // what a warm start continues from besides the cones' states: the scalings of the last solve (the reference
  // keeps them in the program's memory, WorkspaceStats) and whether the states were ever initialised
  std::vector<double> b_scaling, c_scaling;
  bool initialised = false;

  void* s() const { return ctx.stream(); }
  void UploadCoef(size_t offset, size_t count) {
    CudaCheck(cudaMemcpyAsync(coef.get() + offset, hcoef.get() + offset, sizeof(double) * count,
                              cudaMemcpyHostToDevice, ctx.cuda_stream()),
              "H2D coefficients");
  }
  // Columns [first, first + count) of equality block `e` (column j < nvars: column j of A, column nvars: b) from
  // `data`, B host blocks of rows x count column-major, into the constant rows m + offset .. of every program's H
  // (column variables[j]; H[p] is ldh x N) and AQc (b). The cones' Schur kernels assign only the leading m x m block
  // of H and the first m entries of AW / AQc, and the LDL^T leaves H as it is: these survive every Newton step.
  void WriteEqualityColumns(const EqualitySlot& e, int first, int count, const double* data) {
    const int nv = static_cast<int>(e.variables.size());
    for (int j = first; j < first + count; j++) {
      const double* src = data + static_cast<size_t>(j - first) * e.rows;
      double* dst = (j < nv) ? H.get() + static_cast<size_t>(e.variables[j]) * ldh + m + e.offset
                             : AQc.get() + m + e.offset;
      const size_t dpitch = sizeof(double) * ((j < nv) ? static_cast<size_t>(ldh) * N : vstride);
      CudaCheck(cudaMemcpy2DAsync(dst, dpitch, src, sizeof(double) * e.rows * count, sizeof(double) * e.rows, B,
                                  cudaMemcpyHostToDevice, ctx.cuda_stream()),
                "upload of equality data");
    }
    ctx.Synchronize();  // data is pageable
  }
  void UploadMask(size_t offset) {
    CudaCheck(cudaMemcpyAsync(mask.get() + offset, hmask.get() + offset, sizeof(int) * B,
                              cudaMemcpyHostToDevice, ctx.cuda_stream()),
              "H2D mask");
  }
  void DownloadOut(size_t count) {
    CudaCheck(cudaMemcpyAsync(hout.get(), out.get(), sizeof(double) * count, cudaMemcpyDeviceToHost,
                              ctx.cuda_stream()),
              "D2H outputs");
    ctx.Synchronize();
  }
  // The order of DenseKKTSolver::Assemble: the first full cone assigns the leading m x m block of H, AW[0..m),
  // AQc[0..m) and scal, the other full cones add to them. Each subset cone assigns its own block into sub_schur, and
  // one scatter-add adds those blocks in, zeroing the targets first when no cone is full. Rows m..N-1 (the
  // equality blocks) are never touched.
  void Assemble(const int* active) {
    bool first = true;
    for (auto& c : cones) {
      if (!c.variables.empty()) continue;
      DeviceCheck(cxb_small_schur(s(), B, &c.desc, H.get(), ldh, ldh * N, AW.get(), AQc.get(), vstride,
                                  scal.get(), 2, first ? 0 : 1, active),
                  "cxb_small_schur");
      first = false;
    }
    if (subset.empty()) return;
    for (int k : subset) {
      ConeSlot& c = cones[k];
      const long ld = static_cast<long>(Align4(c.m));
      double* g = sub_schur.get() + c.scratch_offset;
      const long ss = static_cast<long>(sub_stride);
      DeviceCheck(cxb_small_schur(s(), B, &c.desc, g, ld, ss, g + ld * c.m, g + ld * (c.m + 1), ss, g + ld * (c.m + 2),
                                  ss, 0, active),
                  "cxb_small_schur");
    }
    DeviceCheck(cxb_small_scatter_schur(s(), B, static_cast<int>(subset.size()), sub_table.get(), gather_idx.get(),
                                        sub_schur.get(), static_cast<long>(sub_stride), m, H.get(), ldh, ldh * N,
                                        AW.get(), AQc.get(), static_cast<long>(vstride), scal.get(), 2, first ? 0 : 1,
                                        active),
                "cxb_small_scatter_schur");
  }
  // The subset cones' slices of x (y or y2) behind its first vstride entries, before a slack pass reads them.
  void Gather(double* x, const int* active) {
    if (gather_count == 0) return;
    DeviceCheck(cxb_small_gather(s(), B, gather_count, gather_idx.get(), x, static_cast<long>(ystride),
                                 static_cast<long>(vstride), active),
                "cxb_small_gather");
  }
  // The KKT factor and solve: Cholesky without multipliers, the regularised LDL^T with them, which never fails
  // (kkt_solver.cc:172-199: the input decides).
  void Factor(const int* active) {
    if (multipliers == 0) {
      DeviceCheck(cxb_small_potrf(s(), B, N, H.get(), ldh, ldh * N, info.get(), active), "cxb_small_potrf");
      return;
    }
    DeviceCheck(cxb_small_ldlt(s(), B, N, H.get(), ldh, ldh * N, L.get(), ldh, ldh * N, perm.get(), N, signs.get(),
                               N, info.get() + 2 * static_cast<size_t>(B), active),
                "cxb_small_ldlt");
  }
  void Solve(double* x, const int* active) {  // x: y or y2 (stride ystride)
    if (multipliers == 0) {
      DeviceCheck(cxb_small_potrs(s(), B, N, H.get(), ldh, ldh * N, x, ystride, active), "cxb_small_potrs");
      return;
    }
    DeviceCheck(cxb_small_ldlt_solve(s(), B, N, L.get(), ldh, ldh * N, perm.get(), N, signs.get(), N, x, ystride,
                                     active),
                "cxb_small_ldlt_solve");
  }
};

BatchProgram::BatchProgram(const std::vector<Program*>& programs) : impl_(std::make_unique<Impl>()) {
  Impl& d = *impl_;
  if (programs.empty()) throw std::runtime_error("conex-b200: empty batch");
  const int B = static_cast<int>(programs.size());
  batch_ = d.B = B;
  m_ = d.m = programs[0]->GetNumberOfVariables();
  const int m = m_;
  // ---- structure of program 0; every other program must match it ------------------------------
  constexpr int kEquality = -1;
  struct Shape {
    int type, n;                 // n: the order of a cone, the rows of an equality block
    std::vector<int> variables;  // equality blocks: the columns of A; cones: their variables, empty when all in order
  };
  auto shape_of = [&](Container& c, Shape* sh) {
    sh->variables.clear();
    if (auto* lp = std::any_cast<LinearConstraint>(&c.obj)) {
      sh->type = CXB_CONE_LP;
      sh->n = lp->order();
    } else if (auto* soc = std::any_cast<SOCConstraint>(&c.obj)) {
      sh->type = CXB_CONE_SOC;
      sh->n = soc->order();
    } else if (auto* lmi = std::any_cast<DenseLMIConstraint>(&c.obj)) {
      sh->type = CXB_CONE_PSD;
      sh->n = lmi->order();
    } else if (auto* eq = std::any_cast<EqualityConstraints>(&c.obj)) {
      // any subset of the variables, followed by the block's multipliers (Program::AddConstraint)
      sh->type = kEquality;
      sh->n = eq->rows();
      const int nv = static_cast<int>(c.variables.size()) - eq->rows();
      if (nv != eq->number_of_columns()) throw std::runtime_error("conex-b200: malformed equality block");
      sh->variables.assign(c.variables.begin(), c.variables.begin() + nv);
      for (int v : sh->variables) {
        if (v < 0 || v >= m) throw std::runtime_error("conex-b200: malformed equality block");
      }
      return;
    } else {
      throw std::runtime_error(
          "conex-b200: batched solves support LP, second-order and dense LMI cones and equality constraints");
    }
    // any list of distinct variables (Program::AddConstraint); 0..m-1 in order is a full cone
    bool full = static_cast<int>(c.variables.size()) == m;
    std::vector<char> seen(m, 0);
    for (size_t i = 0; i < c.variables.size(); i++) {
      const int v = c.variables[i];
      if (v < 0 || v >= m || seen[v]) throw std::runtime_error("conex-b200: malformed variable list of a cone");
      seen[v] = 1;
      full = full && v == static_cast<int>(i);
    }
    if (c.variables.empty()) throw std::runtime_error("conex-b200: a cone without variables");
    if (!full) sh->variables = c.variables;
  };
  std::vector<Shape> shapes;
  for (auto& c : programs[0]->eqs) {
    Shape sh;
    shape_of(c, &sh);
    shapes.push_back(sh);
  }
  const size_t nconstraints = shapes.size();
  for (const Shape& sh : shapes) {
    if (sh.type == kEquality) {
      EqualitySlot e;
      e.rows = sh.n;
      e.offset = d.multipliers;
      e.variables = sh.variables;
      d.multipliers += sh.n;
      d.slot_of.push_back(-1 - static_cast<int>(d.equalities.size()));
      d.equalities.push_back(std::move(e));
    } else {
      d.slot_of.push_back(static_cast<int>(d.cones.size()));
      d.cones.emplace_back();
      d.cones.back().type = sh.type;
      d.cones.back().n = sh.n;
      d.cones.back().variables = sh.variables;
    }
  }
  if (d.cones.empty()) throw std::runtime_error("conex-b200: batched programs have no cones");
  if (programs[0]->NumberOfMultipliers() != d.multipliers) {
    throw std::runtime_error("conex-b200: malformed equality blocks");
  }
  const int N = d.N = m + d.multipliers;
  const size_t nc = d.cones.size();
  d.vstride = Align4(N);
  d.rank = 0;
  // subset cones: their slices of y at 4-aligned offsets behind y, their Schur blocks in one scratch area per program
  std::vector<int> gather_idx, sub_table;
  for (size_t k = 0; k < nc; k++) {
    ConeSlot& c = d.cones[k];
    if (c.variables.empty()) {
      c.m = m;
      continue;
    }
    c.m = static_cast<int>(c.variables.size());
    c.gather_offset = gather_idx.size();
    c.scratch_offset = d.sub_stride;
    sub_table.insert(sub_table.end(), {c.m, static_cast<int>(c.gather_offset), static_cast<int>(c.scratch_offset)});
    gather_idx.insert(gather_idx.end(), c.variables.begin(), c.variables.end());
    gather_idx.resize(Align4(gather_idx.size()), -1);
    d.sub_stride += Align4(c.m) * (c.m + 2) + 4;  // G_k | AW_k | AQc_k | 2 scalars
    d.subset.push_back(static_cast<int>(k));
  }
  d.gather_count = static_cast<int>(gather_idx.size());
  d.ystride = d.vstride + gather_idx.size();
  if (!d.subset.empty()) {
    d.gather_idx.Resize(gather_idx.size());
    d.sub_table.Resize(sub_table.size());
    d.sub_schur.Resize(d.sub_stride * B);
    // pageable sources: they stay alive until the synchronisation after the packing below
    CudaCheck(cudaMemcpyAsync(d.gather_idx.get(), gather_idx.data(), sizeof(int) * gather_idx.size(),
                              cudaMemcpyHostToDevice, d.ctx.cuda_stream()),
              "upload of the subset cones' variables");
    CudaCheck(cudaMemcpyAsync(d.sub_table.get(), sub_table.data(), sizeof(int) * sub_table.size(),
                              cudaMemcpyHostToDevice, d.ctx.cuda_stream()),
              "upload of the subset cones' layout");
  }
  for (size_t k = 0; k < nc; k++) {
    ConeSlot& c = d.cones[k];
    c.rows = c.type == CXB_CONE_LP ? c.n : (c.type == CXB_CONE_SOC ? c.n + 1 : c.n * c.n);
    c.rank = c.type == CXB_CONE_LP ? c.n : (c.type == CXB_CONE_SOC ? 2 : c.n);
    d.rank += c.rank;
    c.state_size = cxb_small_state_size(c.type, c.n);
    c.work_size = cxb_small_work_size(c.type, c.n, c.m);
    const size_t per = static_cast<size_t>(c.rows) * (c.m + 1);
    c.data.Resize(per * B);
    c.state.Resize(c.state_size * B);
    if (c.work_size) c.work.Resize(c.work_size * B);
    c.desc.type = c.type;
    c.desc.n = c.n;
    c.desc.m = c.m;
    c.desc.y_offset = c.variables.empty() ? 0 : static_cast<int>(d.vstride + c.gather_offset);
    c.desc.data = c.data.get();
    c.desc.data_stride = static_cast<long>(per);
    c.desc.state = c.state.get();
    c.desc.state_stride = static_cast<long>(c.state_size);
    c.desc.work = c.work_size ? c.work.get() : nullptr;
    c.desc.work_stride = static_cast<long>(c.work_size);
    c.desc.packed = nullptr;
    c.desc.packed_stride = 0;
  }
  // ---- pack the cone data; gather the equality data on the host --------------------------------------
  const size_t nm = static_cast<size_t>(d.multipliers);
  // per equality block, [A | b] of every program: B blocks of rows x (nvars + 1), as WriteEqualityColumns takes them
  std::vector<std::vector<double>> eq_data(d.equalities.size());
  for (size_t q = 0; q < d.equalities.size(); q++) {
    const EqualitySlot& e = d.equalities[q];
    eq_data[q].resize(static_cast<size_t>(e.rows) * (e.variables.size() + 1) * B);
  }
  for (int p = 0; p < B; p++) {
    Program& prog = *programs[p];
    if (prog.GetNumberOfVariables() != m || prog.NumberOfMultipliers() != d.multipliers ||
        prog.eqs.size() != nconstraints) {
      throw std::runtime_error("conex-b200: programs of a batch must have identical structure");
    }
    size_t k = 0, q = 0;
    for (auto& c : prog.eqs) {
      Shape sh;
      shape_of(c, &sh);
      if (sh.type != shapes[k].type || sh.n != shapes[k].n || sh.variables != shapes[k].variables) {
        throw std::runtime_error("conex-b200: programs of a batch must have identical structure");
      }
      if (sh.type == kEquality) {
        // ConstructSchurComplementSystem(EqualityConstraints*) (equality_constraint.cc:13-30): A on (multipliers,
        // variables), zeros elsewhere in these rows of H, including the multiplier block; b in AQc, zeros in AW
        const EqualitySlot& e = d.equalities[q];
        auto* eq = std::any_cast<EqualityConstraints>(&c.obj);
        const size_t nv = e.variables.size();
        double* block = eq_data[q++].data() + static_cast<size_t>(p) * e.rows * (nv + 1);
        d.ctx.Download(block, eq->device_A(), static_cast<size_t>(e.rows) * nv);
        d.ctx.Download(block + static_cast<size_t>(e.rows) * nv, eq->device_b(), e.rows);
        k++;
        continue;
      }
      ConeSlot& slot = d.cones[d.slot_of[k]];
      const size_t per = static_cast<size_t>(slot.rows) * (slot.m + 1);
      double* dst = slot.data.get() + per * p;
      if (sh.type == CXB_CONE_PSD) {
        auto* lmi = std::any_cast<DenseLMIConstraint>(&c.obj);
        CudaCheck(cudaMemcpyAsync(dst, lmi->device_matrices(), sizeof(double) * per, cudaMemcpyDeviceToDevice,
                                  d.ctx.cuda_stream()),
                  "packing of an LMI block");
      } else {
        const auto& host = (sh.type == CXB_CONE_LP)
                               ? std::any_cast<LinearConstraint>(&c.obj)->host_data()
                               : std::any_cast<SOCConstraint>(&c.obj)->host_data();
        CudaCheck(cudaMemcpyAsync(dst, host.data(), sizeof(double) * per, cudaMemcpyHostToDevice, d.ctx.cuda_stream()),
                  "packing of a small cone");
      }
      k++;
    }
  }
  d.ctx.Synchronize();
  // ---- packed copies of the LMI operators (symmetric matrices: the slack passes read half the bytes) -------------
  {
    DeviceBuffer<int> flags;
    flags.Resize(nc);
    CudaCheck(cudaMemsetAsync(flags.get(), 0, sizeof(int) * nc, d.ctx.cuda_stream()), "memset");
    for (size_t k = 0; k < nc; k++) {
      ConeSlot& c = d.cones[k];
      if (c.type != CXB_CONE_PSD) continue;
      const size_t stride = Align4(static_cast<size_t>(c.m + 1) * (static_cast<size_t>(c.n) * (c.n + 1) / 2));
      c.packed.Resize(stride * B);
      DeviceCheck(cxb_small_pack_symmetric(d.s(), B, &c.desc, c.packed.get(), static_cast<long>(stride),
                                           flags.get() + k),
                  "cxb_small_pack_symmetric");
    }
    std::vector<int> asymmetric(nc, 0);
    d.ctx.DownloadInts(asymmetric.data(), flags.get(), nc);
    for (size_t k = 0; k < nc; k++) {
      ConeSlot& c = d.cones[k];
      if (c.type == CXB_CONE_PSD && !asymmetric[k]) {
        c.desc.packed = c.packed.get();
        c.desc.packed_stride =
            static_cast<long>(Align4(static_cast<size_t>(c.m + 1) * (static_cast<size_t>(c.n) * (c.n + 1) / 2)));
      } else {
        c.packed.Resize(0);
      }
    }
    for (auto& c : d.cones) d.descs.push_back(c.desc);
  }
  // ---- Newton-system storage ------------------------------------------------------------------------
  d.ldh = static_cast<long>(Align4(N));
  d.H.Resize(static_cast<size_t>(d.ldh) * N * B);
  if (d.multipliers) {
    d.L.Resize(static_cast<size_t>(d.ldh) * N * B);
    d.perm.Resize(static_cast<size_t>(N) * B);
    d.signs.Resize(static_cast<size_t>(N) * B);
  }
  d.AW.Resize(d.vstride * B);
  d.AQc.Resize(d.vstride * B);
  d.scal.Resize(2 * static_cast<size_t>(B));
  d.b.Resize(d.vstride * B);
  d.y.Resize(d.ystride * B);
  d.y2.Resize(d.ystride * B);
  d.coef.Resize(5 * static_cast<size_t>(B));
  d.out.Resize(static_cast<size_t>(B) * (4 * nc + 4));
  d.info.Resize((d.multipliers ? 3 : 2) * static_cast<size_t>(B));
  d.mask.Resize(3 * static_cast<size_t>(B));
  d.asymmetric.Resize(1);
  d.hcoef.Reserve(std::max<size_t>(5 * static_cast<size_t>(B), d.vstride * B));
  d.hout.Reserve(std::max<size_t>(static_cast<size_t>(B) * (4 * nc + 4), d.ystride * B));
  d.hinfo.Reserve(2 * static_cast<size_t>(B));
  d.hmask.Reserve(3 * static_cast<size_t>(B));
  d.b_scaling.assign(B, 1.0);
  d.c_scaling.assign(B, 1.0);
  results_.assign(B, BatchResult());
  if (d.multipliers) {
    // rows m..N-1 of every H (H[p] is ldh x N, so column c of program p is column p N + c of one B N-column matrix)
    // and AW[m..N) are zero outside the blocks' A (equality_constraint.cc:13-30, including the multiplier block)
    cudaStream_t cs = d.ctx.cuda_stream();
    CudaCheck(cudaMemset2DAsync(d.H.get() + m, sizeof(double) * d.ldh, 0, sizeof(double) * nm,
                                static_cast<size_t>(N) * B, cs),
              "memset");
    CudaCheck(cudaMemset2DAsync(d.AW.get() + m, sizeof(double) * d.vstride, 0, sizeof(double) * nm, B, cs), "memset");
    for (size_t q = 0; q < d.equalities.size(); q++) {
      const EqualitySlot& e = d.equalities[q];
      d.WriteEqualityColumns(e, 0, static_cast<int>(e.variables.size()) + 1, eq_data[q].data());
    }
  }
}

BatchProgram::~BatchProgram() = default;

int BatchProgram::DualVariableSize(int cone) const {
  const int k = impl_->slot_of.at(cone);
  if (k < 0) return 0;  // an equality block has no dual variable (equality_constraint.h:9-18)
  const ConeSlot& c = impl_->cones.at(k);
  return c.type == CXB_CONE_PSD ? c.n * c.n : c.rows;
}

void BatchProgram::GetDualVariable(int p, int cone, double* host_out) {
  Impl& d = *impl_;
  const int k = d.slot_of.at(cone);
  if (k < 0) return;
  const ConeSlot& c = d.cones.at(k);
  const int sz = DualVariableSize(cone);
  d.ctx.Download(host_out, c.state.get() + c.state_size * p, sz);
  const BatchResult& r = results_.at(p);
  ScaleDualVariable(r.num_iterations, r.primal_infeasible, r.inv_sqrt_mu, r.b_scaling, host_out, sz);
}

bool BatchProgram::ConstraintDataShape(int constraint, int* rows, int* columns) const {
  const Impl& d = *impl_;
  if (constraint < 0 || constraint >= static_cast<int>(d.slot_of.size())) return false;
  const int k = d.slot_of[constraint];
  *rows = k < 0 ? d.equalities[-1 - k].rows : d.cones[k].rows;
  *columns = k < 0 ? static_cast<int>(d.equalities[-1 - k].variables.size()) + 1 : d.cones[k].m + 1;
  return true;
}

void BatchProgram::UpdateConstraintData(int constraint, int first, int count, const double* data) {
  Impl& d = *impl_;
  int rows = 0, columns = 0;
  if (!ConstraintDataShape(constraint, &rows, &columns)) {
    throw std::runtime_error("conex-b200: no such constraint in the batch");
  }
  const int k = d.slot_of[constraint];
  if (first < 0 || count < 1 || count > columns - first || !data) {
    throw std::runtime_error("conex-b200: bad column range or data for a constraint update");
  }
  if (k < 0) {
    d.WriteEqualityColumns(d.equalities[-1 - k], first, count, data);
    return;
  }
  ConeSlot& c = d.cones[k];
  const size_t width = sizeof(double) * rows * count;
  CudaCheck(cudaMemcpy2DAsync(c.data.get() + static_cast<size_t>(first) * rows, sizeof(double) * c.desc.data_stride,
                              data, width, width, d.B, cudaMemcpyHostToDevice, d.ctx.cuda_stream()),
            "upload of constraint data");
  if (c.desc.packed) {
    // refresh the packed lower triangles of the changed matrices; data that is not symmetric drops the packed copy
    // for good, as at construction
    CudaCheck(cudaMemsetAsync(d.asymmetric.get(), 0, sizeof(int), d.ctx.cuda_stream()), "memset");
    DeviceCheck(cxb_small_pack_symmetric_columns(d.s(), d.B, &c.desc, first, count, c.packed.get(),
                                                 c.desc.packed_stride, d.asymmetric.get()),
                "cxb_small_pack_symmetric_columns");
    int asymmetric = 0;
    d.ctx.DownloadInts(&asymmetric, d.asymmetric.get(), 1);
    if (asymmetric) {
      c.desc.packed = nullptr;
      c.desc.packed_stride = 0;
      c.packed.Resize(0);
      d.descs[k] = c.desc;
    }
  }
  d.ctx.Synchronize();  // data is pageable
}

int BatchProgram::Maximize(const double* b_in, const SolverConfiguration& cfg, double* y_out) {
  Impl& d = *impl_;
  const int B = batch_, m = m_, N = d.N;
  const size_t nc = d.cones.size();
  const size_t vs = d.vstride;
  const size_t ys = d.ystride;  // y and y2
  const bool warm = cfg.initialization_mode != CONEX_INITIALIZATION_MODE_COLDSTART;
  if (warm && !d.initialised) {
    throw std::runtime_error("conex-b200: a warm start needs a previous solve of the batch");
  }
  if (cfg.kkt_solver == CONEX_QR_FACTORIZATION) {
    throw std::runtime_error("conex-b200: the QR KKT mode is not implemented on the device");
  }
  if (d.multipliers > 0 && cfg.iterative_refinement_iterations > 0) {
    throw std::runtime_error(
        "conex-b200: iterative refinement is not implemented for batched programs with equality constraints");
  }
  if (cfg.enable_line_search) {
    // the reference runs a line search when every constraint is an LP cone or an equality block
    // (cone_program.h:211-216); `cones` holds no equality blocks
    bool lp_only = true;
    for (const auto& c : d.cones) lp_only = lp_only && (c.type == CXB_CONE_LP);
    if (lp_only) {
      throw std::runtime_error(
          "conex-b200: enable_line_search on programs of LP cones and equality constraints only is not implemented");
    }
  }
  void* s = d.s();
  cudaStream_t cs = d.ctx.cuda_stream();
  std::vector<NewtonControl> st;
  results_.assign(B, BatchResult());
  step_ms_.clear();

  // ---- cost vectors; a cold start resets the scalings and the cones (cone_program.cc:350-354) ------------
  for (int p = 0; p < B; p++) {
    const double* bp = b_in + static_cast<size_t>(p) * m;
    for (int i = 0; i < m; i++) d.hcoef[p * vs + i] = bp[i];
    for (size_t i = m; i < vs; i++) d.hcoef[p * vs + i] = 0;
    st.emplace_back(cfg, d.rank, bp, m, warm ? d.b_scaling[p] : 1.0, warm ? d.c_scaling[p] : 1.0);
  }
  CudaCheck(cudaMemcpyAsync(d.b.get(), d.hcoef.get(), sizeof(double) * vs * B, cudaMemcpyHostToDevice, cs),
            "H2D cost vectors");
  d.ctx.Synchronize();  // hcoef is reused below
  d.ctx.Zero(d.y.get(), ys * B);
  const int ncones = static_cast<int>(nc);
  if (!warm) {
    DeviceCheck(cxb_small_set_identity_multi(s, B, ncones, d.descs.data(), nullptr), "cxb_small_set_identity_multi");
    d.initialised = true;
  }
  cudaEvent_t ev_begin, ev_end, ev_a, ev_b;
  CudaCheck(cudaEventCreate(&ev_begin), "cudaEventCreate");
  CudaCheck(cudaEventCreate(&ev_end), "cudaEventCreate");
  CudaCheck(cudaEventCreate(&ev_a), "cudaEventCreate");
  CudaCheck(cudaEventCreate(&ev_b), "cudaEventCreate");
  CudaCheck(cudaEventRecord(ev_begin, cs), "cudaEventRecord");

  int* active = d.mask.get();
  int* mu_mask = d.mask.get() + B;
  int* abort_mask = d.mask.get() + 2 * static_cast<size_t>(B);
  double* coef_a = d.coef.get();
  double* coef_b = d.coef.get() + B;
  double* coef_c = d.coef.get() + 2 * static_cast<size_t>(B);
  double* coef_cw = d.coef.get() + 3 * static_cast<size_t>(B);
  double* coef_step = d.coef.get() + 4 * static_cast<size_t>(B);
  double* cone_out = d.out.get();                                   // B x nc x 4
  double* dots = d.out.get() + static_cast<size_t>(B) * 4 * nc;     // B x 4
  const long ostride = static_cast<long>(4 * nc);

  for (int i = 0; i < cfg.max_iterations; i++) {
    // ---- loop control of every program (reference cone_program.cc:312-336) -----------------------
    int nactive = 0;
    bool new_scalings = false;
    for (int p = 0; p < B; p++) {
      d.hmask[p] = st[p].Begin(i);
      nactive += d.hmask[p];
      new_scalings = new_scalings || (d.hmask[p] && st[p].NeedsAqcNorm());
    }
    if (nactive == 0) break;
    d.UploadMask(0);
    CudaCheck(cudaEventRecord(ev_a, cs), "cudaEventRecord");

    // ---- assemble, (rescale,) factor ---------------------------------------------------------------
    d.Assemble(active);
    if (new_scalings) {
      DeviceCheck(cxb_batched_dot(s, B, N, d.AQc.get(), vs, d.AQc.get(), vs, dots, 4), "cxb_batched_dot");
    }
    d.Factor(active);
    if (!d.multipliers) {
      CudaCheck(cudaMemcpyAsync(d.hinfo.get(), d.info.get(), sizeof(int) * B, cudaMemcpyDeviceToHost, cs),
                "D2H info");
    }
    if (new_scalings) {
      CudaCheck(cudaMemcpyAsync(d.hout.get(), dots, sizeof(double) * 4 * B, cudaMemcpyDeviceToHost, cs), "D2H norms");
    }
    d.ctx.Synchronize();
    bool mask_changed = false;
    bool any_mu = false;
    bool any_restart = false;
    for (int p = 0; p < B; p++) {
      NewtonControl& q = st[p];
      d.hmask[B + p] = 0;
      d.hmask[2 * static_cast<size_t>(B) + p] = 0;
      if (!q.stepping()) continue;
      q.Rescale(new_scalings ? d.hout[4 * p] : 0.0);
      if (!d.multipliers && d.hinfo[p] != 0) {
        d.hmask[p] = 0;
        mask_changed = true;
        if (q.RestartOnFactorizationFailure()) {
          d.hmask[2 * static_cast<size_t>(B) + p] = 1;
          any_restart = true;
        }
        continue;
      }
      if (q.update_mu()) {
        d.hmask[B + p] = 1;
        any_mu = true;
      }
    }
    if (mask_changed) d.UploadMask(0);
    if (any_restart) {
      d.UploadMask(2 * static_cast<size_t>(B));
      DeviceCheck(cxb_small_set_identity_multi(s, B, ncones, d.descs.data(), abort_mask),
                  "cxb_small_set_identity_multi");
    }

    // ---- mu from the divergence bound (reference cone_program.cc:173-214) --------------------------
    if (any_mu) {
      d.UploadMask(B);
      for (int p = 0; p < B; p++) {
        d.hcoef[p] = st[p].c_scaling();
        d.hcoef[B + p] = -st[p].b_scaling();
        d.hcoef[3 * static_cast<size_t>(B) + p] = st[p].c_scaling();
      }
      d.UploadCoef(0, 2 * static_cast<size_t>(B));
      d.UploadCoef(3 * static_cast<size_t>(B), B);
      DeviceCheck(cxb_batched_lincomb(s, B, N, coef_a, d.AQc.get(), vs, coef_b, d.b.get(), vs, nullptr, nullptr, 0,
                                      d.y.get(), ys, mu_mask),
                  "cxb_batched_lincomb");
      d.Solve(d.y.get(), mu_mask);
      d.Gather(d.y.get(), mu_mask);
      DeviceCheck(cxb_small_eigen_multi(s, B, ncones, d.descs.data(), d.y.get(), ys, 0.0, coef_cw, cone_out, ostride,
                                        mu_mask),
                  "cxb_small_eigen_multi");
      d.DownloadOut(static_cast<size_t>(B) * 4 * nc);
    }
    for (int p = 0; p < B; p++) {
      NewtonControl& q = st[p];
      if (!q.stepping()) continue;
      SlackEigenvalueSum w;
      for (size_t k = 0; k < nc && q.NeedsEigenvalues(); k++) {
        const double* o = d.hout.get() + (static_cast<size_t>(p) * nc + k) * 4;
        w.Add(o[0], o[1], o[2], o[3]);
      }
      q.ChooseK(w);
      d.hcoef[p] = q.k() * q.b_scaling();
      d.hcoef[B + p] = q.k() * q.c_scaling();
      d.hcoef[2 * static_cast<size_t>(B) + p] = -2.0;
      d.hcoef[3 * static_cast<size_t>(B) + p] = q.k() * q.c_scaling();
    }

    // ---- Newton direction: y = H^{-1} (k (b b_s + AQc c_s) - 2 AW) (cone_program.cc:409-414) ------
    d.UploadCoef(0, 4 * static_cast<size_t>(B));
    DeviceCheck(cxb_batched_lincomb(s, B, N, coef_a, d.b.get(), vs, coef_b, d.AQc.get(), vs, coef_c, d.AW.get(), vs,
                                    d.y.get(), ys, active),
                "cxb_batched_lincomb");
    d.Solve(d.y.get(), active);
    d.Gather(d.y.get(), active);
    DeviceCheck(cxb_small_prepare_multi(s, B, ncones, d.descs.data(), d.y.get(), ys, 0, 0.0, coef_cw, 1.0, cone_out,
                                        ostride, active),
                "cxb_small_prepare_multi");
    d.DownloadOut(static_cast<size_t>(B) * 4 * nc);
    bool any_abort = false;
    for (int p = 0; p < B; p++) {
      NewtonControl& q = st[p];
      d.hcoef[4 * static_cast<size_t>(B) + p] = 1.0;
      d.hmask[2 * static_cast<size_t>(B) + p] = 0;
      if (!q.stepping()) continue;
      double ninf = -1, nsq = 0;
      for (size_t k = 0; k < nc; k++) {
        const double* o = d.hout.get() + (static_cast<size_t>(p) * nc + k) * 4;
        ninf = std::max(ninf, o[0]);
        nsq += o[1];
      }
      if (!q.Step(ninf, nsq, &d.hcoef[4 * static_cast<size_t>(B) + p])) {
        d.hmask[p] = 0;
        d.hmask[2 * static_cast<size_t>(B) + p] = 1;
        any_abort = true;
      }
    }
    d.UploadCoef(4 * static_cast<size_t>(B), B);
    if (any_abort) {
      d.UploadMask(0);
      d.UploadMask(2 * static_cast<size_t>(B));
      DeviceCheck(cxb_small_set_identity_multi(s, B, ncones, d.descs.data(), abort_mask),
                  "cxb_small_set_identity_multi");
    }
    DeviceCheck(cxb_small_take_step_multi(s, B, ncones, d.descs.data(), 1.0, coef_step, 1.0, d.info.get() + B, active),
                "cxb_small_take_step_multi");
    // ---- objectives (cone_program.cc:441-467) -------------------------------------------------------
    DeviceCheck(cxb_batched_dot(s, B, N, d.b.get(), vs, d.y.get(), ys, dots + 0, 4), "cxb_batched_dot");
    DeviceCheck(cxb_batched_dot(s, B, N, d.AQc.get(), vs, d.y.get(), ys, dots + 1, 4), "cxb_batched_dot");
    CudaCheck(cudaEventRecord(ev_b, cs), "cudaEventRecord");
    CudaCheck(cudaMemcpyAsync(d.hout.get(), dots, sizeof(double) * 4 * B, cudaMemcpyDeviceToHost, cs), "D2H dots");
    CudaCheck(cudaMemcpyAsync(d.hout.get() + 4 * static_cast<size_t>(B), d.scal.get(), sizeof(double) * 2 * B,
                              cudaMemcpyDeviceToHost, cs),
              "D2H scalars");
    d.ctx.Synchronize();
    float ms = 0;
    cudaEventElapsedTime(&ms, ev_a, ev_b);
    step_ms_.push_back(ms);
    for (int p = 0; p < B; p++) {
      if (!st[p].stepping()) continue;
      const double* sc = d.hout.get() + 4 * static_cast<size_t>(B) + 2 * p;
      st[p].End(d.hout[4 * p + 0], d.hout[4 * p + 1], sc[0], sc[1]);
    }
  }

  // ---- results (cone_program.cc:486-530) -------------------------------------------------------------
  CudaCheck(cudaMemcpyAsync(d.hout.get(), d.y.get(), sizeof(double) * ys * B, cudaMemcpyDeviceToHost, cs), "D2H y");
  d.ctx.Synchronize();
  int solved_count = 0;
  bool any_recover = false;
  for (int p = 0; p < B; p++) {
    const NewtonControl& q = st[p];
    BatchResult& r = results_[p];
    r.by = q.by();
    r.cx = q.cx();
    r.inv_sqrt_mu = q.k();
    r.b_scaling = d.b_scaling[p] = q.b_scaling();
    r.c_scaling = d.c_scaling[p] = q.c_scaling();
    r.d_inf = q.d_inf();
    double* yp = y_out + static_cast<size_t>(p) * m;
    for (int j = 0; j < m; j++) yp[j] = d.hout[p * ys + j];
    static_cast<ConexStatus&>(r) = q.Finish(yp, m);
    solved_count += r.solved;
    d.hmask[p] = !q.failed();
    any_recover = any_recover || !q.failed();
  }
  if (cfg.prepare_dual_variables && any_recover) {
    // reference cone_program.cc:500-516
    d.UploadMask(0);
    d.Assemble(active);
    d.Factor(active);
    for (int p = 0; p < B; p++) {
      d.hcoef[p] = st[p].k() * st[p].b_scaling();
      d.hcoef[B + p] = -1.0;
    }
    d.UploadCoef(0, 2 * static_cast<size_t>(B));
    DeviceCheck(cxb_batched_lincomb(s, B, N, coef_a, d.b.get(), vs, coef_b, d.AW.get(), vs, nullptr, nullptr, 0,
                                    d.y2.get(), ys, active),
                "cxb_batched_lincomb");
    d.Solve(d.y2.get(), active);
    d.Gather(d.y2.get(), active);
    DeviceCheck(cxb_small_prepare_multi(s, B, ncones, d.descs.data(), d.y2.get(), ys, 1, 0.0, nullptr, 0.0, cone_out,
                                        ostride, active),
                "cxb_small_prepare_multi");
  }
  CudaCheck(cudaEventRecord(ev_end, cs), "cudaEventRecord");
  d.ctx.Synchronize();
  float total = 0;
  cudaEventElapsedTime(&total, ev_begin, ev_end);
  total_ms_ = total;
  cudaEventDestroy(ev_begin);
  cudaEventDestroy(ev_end);
  cudaEventDestroy(ev_a);
  cudaEventDestroy(ev_b);
  return solved_count;
}

}  // namespace conex

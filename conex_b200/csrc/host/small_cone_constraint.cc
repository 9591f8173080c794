#include "small_cone_constraint.h"

#include <algorithm>

namespace conex {

struct SmallConeConstraint::Device {
  DeviceBuffer<double> data;  // rows x (m + 1)
  DeviceBuffer<double> work;
  DeviceBuffer<int> info;
  bool dirty = true;          // host copy changed since the last upload
};

SmallConeConstraint::SmallConeConstraint(int type, int n, int m, const double* A, const double* c)
    : type_(type), n_(n), m_(m), rows_(type == CXB_CONE_SOC ? n + 1 : n), workspace_(type, n),
      host_(std::make_shared<std::vector<double>>(static_cast<size_t>(rows_) * (m + 1), 0.0)),
      dev_(std::make_shared<Device>()) {
  if (A) std::copy(A, A + static_cast<size_t>(rows_) * m, host_->begin());
  if (c) std::copy(c, c + rows_, host_->begin() + static_cast<size_t>(rows_) * m);
}

cxb_small_cone SmallConeConstraint::Descriptor() {
  Device& d = *dev_;
  if (d.dirty) {
    d.data.Reserve(host_->size());
    // pageable source: the copy is complete (staged) when cudaMemcpy returns
    CudaCheck(cudaMemcpy(d.data.get(), host_->data(), sizeof(double) * host_->size(), cudaMemcpyHostToDevice),
              "upload of a small cone");
    d.work.Reserve(std::max<size_t>(1, cxb_small_work_size(type_, n_, m_)));
    d.info.Reserve(4);
    d.dirty = false;
  }
  cxb_small_cone c;
  c.type = type_;
  c.n = n_;
  c.m = m_;
  c.y_offset = 0;
  c.data = d.data.get();
  c.data_stride = 0;
  c.state = workspace_.state;
  c.state_stride = 0;
  c.work = d.work.get();
  c.work_stride = 0;
  c.packed = nullptr;
  c.packed_stride = 0;
  return c;
}

void SetIdentity(SmallConeConstraint* o) {
  const cxb_small_cone c = o->Descriptor();
  DeviceCheck(cxb_small_set_identity(o->ctx_->stream(), 1, &c, nullptr), "cxb_small_set_identity");
}

void ConstructSchurComplementSystem(SmallConeConstraint* o, bool initialize, SchurComplementSystem* sys) {
  const cxb_small_cone c = o->Descriptor();
  DeviceCheck(cxb_small_schur(o->ctx_->stream(), 1, &c, sys->G.data, sys->G.ld, 0, sys->AW, sys->AQc, 0,
                              sys->scalars, 0, initialize ? 0 : 1, nullptr),
              "cxb_small_schur");
}

void PrepareStep(SmallConeConstraint* o, const StepOptions& opt, const Ref& y, StepInfo* info) {
  const cxb_small_cone c = o->Descriptor();
  double* out = o->ctx_->scalars() + 8;
  DeviceCheck(cxb_small_prepare(o->ctx_->stream(), 1, &c, y.data, 0, opt.affine ? 1 : 0, opt.c_weight, nullptr,
                                opt.e_weight, out, 0, nullptr),
              "cxb_small_prepare");
  double h[2];
  o->ctx_->Download(h, out, 2);
  info->norminfd = h[0];
  info->normsqrd = h[1];
}

bool TakeStep(SmallConeConstraint* o, const StepOptions& opt) {
  const cxb_small_cone c = o->Descriptor();
  DeviceCheck(cxb_small_take_step(o->ctx_->stream(), 1, &c, opt.step_size, nullptr, opt.e_weight,
                                  o->dev_->info.get(), nullptr),
              "cxb_small_take_step");
  return true;
}

void GetWeightedSlackEigenvalues(SmallConeConstraint* o, const Ref& y, double c_weight,
                                 WeightedSlackEigenvalues* p) {
  const cxb_small_cone c = o->Descriptor();
  double* out = o->ctx_->scalars() + 8;
  DeviceCheck(cxb_small_eigen(o->ctx_->stream(), 1, &c, y.data, 0, c_weight, nullptr, out, 0, nullptr),
              "cxb_small_eigen");
  double h[4];
  o->ctx_->Download(h, out, 4);
  p->lambda_min = h[0];
  p->lambda_max = h[1];
  p->frobenius_norm_squared = h[2];
  p->trace = h[3];
}

bool UpdateLinearOperator(SmallConeConstraint* o, double val, int var, int r, int c, int dim) {
  const bool lp = o->type_ == CXB_CONE_LP;
  CONEX_DEMAND(dim == 0, (lp ? "Complex linear constraints not supported."
                             : "Complex second-order cone not supported."));
  CONEX_DEMAND(c == 0, (lp ? "Linear constraint is not matrix valued."
                           : "Second-order constraint is not matrix valued."));
  CONEX_DEMAND(r < o->rows_, "Row index out of bounds.");
  CONEX_DEMAND((var >= 0) && (r >= 0), "Indices cannot be negative.");
  CONEX_DEMAND(var < o->m_, "Variable index out of bounds.");
  (*o->host_)[static_cast<size_t>(var) * o->rows_ + r] = val;
  o->dev_->dirty = true;
  return false;  // CONEX_SUCCESS
}

bool UpdateAffineTerm(SmallConeConstraint* o, double val, int r, int c, int dim) {
  const bool lp = o->type_ == CXB_CONE_LP;
  CONEX_DEMAND(dim == 0, (lp ? "Complex linear cone not supported." : "Complex second-order cone not supported."));
  CONEX_DEMAND(c == 0, (lp ? "Linear constraint is not matrix valued."
                           : "Second-order constraint is not matrix valued."));
  CONEX_DEMAND(r < o->rows_, "Row index out of bounds.");
  CONEX_DEMAND(r >= 0, "Indices cannot be negative.");
  (*o->host_)[static_cast<size_t>(o->m_) * o->rows_ + r] = val;
  o->dev_->dirty = true;
  return false;
}

}  // namespace conex

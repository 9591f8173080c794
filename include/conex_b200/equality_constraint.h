// Equality constraints A x = b as a "cone" of rank 0 whose multipliers are extra unknowns of the
// KKT system — counterpart of the reference's EqualityConstraints (conex/equality_constraint.{h,cc})
// and of ConstraintManager::AddEqualityConstraint (conex/constraint_manager.h:71-94). Its presence
// switches the KKT solver from Cholesky to the regularised LDL^T (kkt_solver.cc:172-199).
#pragma once
#include <memory>
#include <vector>

#include "constraint.h"

namespace conex {

struct WorkspaceEqualityConstraints {
  friend size_t SizeOf(const WorkspaceEqualityConstraints&) { return 0; }
  friend void Initialize(WorkspaceEqualityConstraints*, double*) {}
  Ref W;  // empty (equality_constraint.h:9-18)
};

class EqualityConstraints {
 public:
  // A: rows x nv column-major (host), b: rows.
  EqualityConstraints(int rows, int nv, const double* A, const double* b);
  int SizeOfDualVariable() const { return rows_; }
  WorkspaceEqualityConstraints* workspace() { return &workspace_; }
  int number_of_variables() const { return 0; }  // equality_constraint.h:46
  void bind(DeviceContext* ctx) { ctx_ = ctx; }
  // Read-only views of the data (the batched solver writes it into its KKT matrices): A is rows x
  // number_of_columns() column-major, b has rows entries; both in device memory.
  int rows() const { return rows_; }
  int number_of_columns() const { return nv_; }
  const double* device_A() const { return dev_->A.get(); }
  const double* device_b() const { return dev_->b.get(); }

  friend int Rank(const EqualityConstraints&) { return 0; }
  friend void SetIdentity(EqualityConstraints*) {}
  friend void ConstructSchurComplementSystem(EqualityConstraints* o, bool initialize,
                                             SchurComplementSystem* sys);
  friend void PrepareStep(EqualityConstraints*, const StepOptions&, const Ref&, StepInfo* info) {
    info->normsqrd = 0;  // equality_constraint.cc:30-35 (the multipliers stay in y)
    info->norminfd = 0;
  }
  friend bool TakeStep(EqualityConstraints*, const StepOptions&) { return true; }
  friend void GetWeightedSlackEigenvalues(EqualityConstraints*, const Ref&, double,
                                          WeightedSlackEigenvalues*) {}

 private:
  struct Device {
    DeviceBuffer<double> A, b;
  };
  int rows_, nv_;
  WorkspaceEqualityConstraints workspace_;
  std::shared_ptr<Device> dev_;
  DeviceContext* ctx_ = nullptr;
};

}  // namespace conex

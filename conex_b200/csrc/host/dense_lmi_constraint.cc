#include "dense_lmi_constraint.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdlib>

#include "../../../include/conex_b200_device.h"
#include "communicator.h"
#include "tridiagonal_eigenvalues.h"

namespace conex {

// Device-side buffers owned by one LMI block. Shared between copies of the constraint object
// (the plugin concept requires copy-constructible types, reference cone_program.h:47-57).
struct DenseLMIConstraint::Storage {
  DeviceBuffer<double> Aall;     // n^2 x (m+1): constraint matrices then C
  DeviceBuffer<double> B;        // n^2 x (m+2): W A_i W, W C W, W        (K1 output / K2 operand)
  DeviceBuffer<double> X;        // symmetric form: packed L^T A_i L, L^T C L, I  ((m+2) x packed size)
  DeviceBuffer<double> Lw;       // symmetric form: Cholesky factor of W
  DeviceBuffer<unsigned char> slices;  // symmetric form: int8 slices of X for the emulated Gram (empty: DMMA Gram)
  bool symmetric = false;        // assemble through cxb_schur_dense_lmi_sym
  DeviceBuffer<double> T;        // panel scratch for A_i W
  DeviceBuffer<double> scratch;  // Lanczos / Padé / LU work
  DeviceBuffer<double> coef;     // [y; -k] for the slack GEMV
  DeviceBuffer<double> small;    // alpha | beta | reductions
  DeviceBuffer<int> iwork;       // LU pivots + permutation, Lanczos count, LU info
  // entry-sparse operator
  bool sparse = false;
  int npos = 0;
  DeviceBuffer<int> sp_offsets, sp_rows, sp_cols, sp_pos_ptr, sp_pos_var;
  DeviceBuffer<long> sp_pos_index;
  DeviceBuffer<double> sp_vals, sp_pos_val, Cdense, sp_work;
  DeviceBuffer<double> rstart;   // Hermitian rule: the random Lanczos start vector
  int panel = 0;
  bool streamed = false;         // B holds one row panel only (cxb_schur_dense_lmi_streamed)
  // sharded blocks only
  DeviceBuffer<double> Hloc;     // (m_local+2) x (m_local+1) augmented Gram of the local diagonal block
  DeviceBuffer<double> recv[2];  // double-buffered chunks of a peer's constraint matrices
  int chunk = 0;                 // constraint matrices per exchanged chunk
  cudaStream_t comm_stream = nullptr;
  cudaEvent_t arrived[2] = {nullptr, nullptr};
  cudaEvent_t consumed[2] = {nullptr, nullptr};
  cudaEvent_t start = nullptr;
  // Peer memory (CUDA IPC over NVLink): peer_x[p] = rank p's packed scaled matrices X mapped into this process, so
  // that a chunk is PULLED by a copy engine straight from the peer's HBM instead of travelling through
  // ncclSend / ncclRecv (measured at 2 GPUs: 122 GB/s through NCCL's point-to-point channels, the exchange stalled
  // the contractions for 10 % of the assembly, profiles/r02_f_bench_c2_2gpu.json). ipc_ready: agreed on by all ranks.
  std::vector<double*> peer_x;
  bool ipc_ready = false;
  DeviceBuffer<int> ipc_words;
  // timing of the last sharded assembly (CUDA events on the compute stream): begin, local block done, before the
  // all-reduce, end; per exchanged chunk: before the wait for its arrival, after it, after its contraction
  cudaEvent_t t_mark[4] = {nullptr, nullptr, nullptr, nullptr};
  std::vector<cudaEvent_t> t_chunk;
  size_t t_chunks_used = 0;
  ~Storage() {
    for (double* p : peer_x) if (p) cudaIpcCloseMemHandle(p);
    for (auto e : t_mark) if (e) cudaEventDestroy(e);
    for (auto e : t_chunk) if (e) cudaEventDestroy(e);
    for (auto e : arrived) if (e) cudaEventDestroy(e);
    for (auto e : consumed) if (e) cudaEventDestroy(e);
    if (start) cudaEventDestroy(start);
    if (comm_stream) cudaStreamDestroy(comm_stream);
  }
};

namespace {
size_t Sq(int n) { return static_cast<size_t>(n) * n; }
}  // namespace

DenseLMIConstraint::DenseLMIConstraint(int n, int m, const double* A, const double* C)
    : n_(n), m_(m), m_local_(m), workspace_(n), data_(std::make_shared<Storage>()) {
  data_->Aall.Resize(Sq(n) * (m + 1));
  CudaCheck(cudaMemcpy(data_->Aall.get(), A, sizeof(double) * Sq(n) * m, cudaMemcpyHostToDevice),
            "upload of LMI matrices");
  CudaCheck(cudaMemcpy(data_->Aall.get() + Sq(n) * m, C, sizeof(double) * Sq(n),
                       cudaMemcpyHostToDevice),
            "upload of LMI affine term");
}

DenseLMIConstraint::DenseLMIConstraint(int n, int m_global, Sharded, DevicePointers dev)
    : n_(n), m_(m_global), workspace_(n), data_(std::make_shared<Storage>()) {
  const Communicator& comm = Communicator::Get();
  if (m_global < comm.world()) {
    throw std::runtime_error("conex-b200: a sharded LMI block needs at least one matrix per rank");
  }
  row_begin_ = ShardBegin(m_global, comm.world(), comm.rank());
  m_local_ = ShardBegin(m_global, comm.world(), comm.rank() + 1) - row_begin_;
  sharded_ = comm.distributed();
  data_->Aall.Resize(Sq(n) * (m_local_ + 1));
  CudaCheck(cudaMemcpy(data_->Aall.get(), dev.A, sizeof(double) * Sq(n) * m_local_,
                       cudaMemcpyDeviceToDevice),
            "copy of LMI matrices");
  CudaCheck(cudaMemcpy(data_->Aall.get() + Sq(n) * m_local_, dev.C, sizeof(double) * Sq(n),
                       cudaMemcpyDeviceToDevice),
            "copy of LMI affine term");
}

DenseLMIConstraint::DenseLMIConstraint(int n, int m_global, Sharded, Uninitialized)
    : n_(n), m_(m_global), workspace_(n), data_(std::make_shared<Storage>()) {
  const Communicator& comm = Communicator::Get();
  if (m_global < comm.world()) {
    throw std::runtime_error("conex-b200: a sharded LMI block needs at least one matrix per rank");
  }
  row_begin_ = ShardBegin(m_global, comm.world(), comm.rank());
  m_local_ = ShardBegin(m_global, comm.world(), comm.rank() + 1) - row_begin_;
  sharded_ = comm.distributed();
  data_->Aall.Resize(Sq(n) * (m_local_ + 1));
}

double* DenseLMIConstraint::mutable_device_matrices() { return data_->Aall.get(); }

DenseLMIConstraint::DenseLMIConstraint(int n, int m, DevicePointers dev)
    : n_(n), m_(m), m_local_(m), workspace_(n), data_(std::make_shared<Storage>()) {
  data_->Aall.Resize(Sq(n) * (m + 1));
  CudaCheck(cudaMemcpy(data_->Aall.get(), dev.A, sizeof(double) * Sq(n) * m, cudaMemcpyDeviceToDevice),
            "copy of LMI matrices");
  CudaCheck(cudaMemcpy(data_->Aall.get() + Sq(n) * m, dev.C, sizeof(double) * Sq(n),
                       cudaMemcpyDeviceToDevice),
            "copy of LMI affine term");
}

const double* DenseLMIConstraint::device_matrices() const { return data_->Aall.get(); }

DenseLMIConstraint::DenseLMIConstraint(int n, int m, EntrySparse)
    : n_(n), m_(m), m_local_(m), workspace_(n), data_(std::make_shared<Storage>()) {}

bool DenseLMIConstraint::entry_sparse() const { return data_->sparse; }

bool DenseLMIConstraint::shard_phase_milliseconds(double* out4) const {
  const Storage& d = *data_;
  if (!sharded_ || d.t_mark[3] == nullptr || cudaEventSynchronize(d.t_mark[3]) != cudaSuccess) return false;
  float local = 0, allreduce = 0, stall = 0, offdiag = 0;
  cudaEventElapsedTime(&local, d.t_mark[0], d.t_mark[1]);
  cudaEventElapsedTime(&allreduce, d.t_mark[2], d.t_mark[3]);
  for (size_t c = 0; c < d.t_chunks_used; c++) {
    float a = 0, b = 0;
    cudaEventElapsedTime(&a, d.t_chunk[3 * c], d.t_chunk[3 * c + 1]);
    cudaEventElapsedTime(&b, d.t_chunk[3 * c + 1], d.t_chunk[3 * c + 2]);
    stall += a;
    offdiag += b;
  }
  out4[0] = local;
  out4[1] = stall;
  out4[2] = offdiag;
  out4[3] = allreduce;
  return true;
}

int DenseLMIConstraint::assembly_form() const {
  const Storage& d = *data_;
  if (d.panel == 0) return 0;  // not decided yet (EnsureScratch runs at the first assembly)
  if (d.sparse) return 4;
  if (d.symmetric) return 3;
  return d.streamed ? 2 : 1;
}

namespace {
template <typename T>
void UploadVector(DeviceBuffer<T>* dst, const std::vector<T>& src) {
  dst->Resize(std::max<size_t>(1, src.size()));
  if (!src.empty()) {
    CudaCheck(cudaMemcpy(dst->get(), src.data(), sizeof(T) * src.size(), cudaMemcpyHostToDevice), "upload");
  }
}
}  // namespace

void DenseLMIConstraint::LoadEntries(const std::vector<Entry>& lower, const double* C) {
  Storage& d = *data_;
  const int n = n_;
  // (1) per-matrix lists with both triangles explicit
  std::vector<int> offsets(m_ + 1, 0), rows, cols;
  std::vector<double> vals;
  std::vector<std::vector<Entry>> by_var(m_);
  for (const Entry& e : lower) by_var[e.var].push_back(e);
  // (2) the same entries grouped by position for the slack
  std::map<long, std::vector<std::pair<int, double>>> by_pos;
  for (int i = 0; i < m_; i++) {
    for (const Entry& e : by_var[i]) {
      rows.push_back(e.r);
      cols.push_back(e.c);
      vals.push_back(e.val);
      by_pos[static_cast<long>(e.c) * n + e.r].push_back({i, e.val});
      if (e.r != e.c) {
        rows.push_back(e.c);
        cols.push_back(e.r);
        vals.push_back(e.val);
        by_pos[static_cast<long>(e.r) * n + e.c].push_back({i, e.val});
      }
    }
    offsets[i + 1] = static_cast<int>(rows.size());
  }
  std::vector<int> pos_ptr(1, 0), pos_var;
  std::vector<long> pos_index;
  std::vector<double> pos_val;
  for (const auto& kv : by_pos) {
    pos_index.push_back(kv.first);
    for (const auto& ve : kv.second) {
      pos_var.push_back(ve.first);
      pos_val.push_back(ve.second);
    }
    pos_ptr.push_back(static_cast<int>(pos_var.size()));
  }
  d.npos = static_cast<int>(pos_index.size());
  UploadVector(&d.sp_offsets, offsets);
  UploadVector(&d.sp_rows, rows);
  UploadVector(&d.sp_cols, cols);
  UploadVector(&d.sp_vals, vals);
  UploadVector(&d.sp_pos_ptr, pos_ptr);
  UploadVector(&d.sp_pos_index, pos_index);
  UploadVector(&d.sp_pos_var, pos_var);
  UploadVector(&d.sp_pos_val, pos_val);
  d.Cdense.Resize(Sq(n));
  CudaCheck(cudaMemcpy(d.Cdense.get(), C, sizeof(double) * Sq(n), cudaMemcpyHostToDevice), "upload of C");
  d.sp_work.Resize(2 * Sq(n));
  if (!d.sparse) d.panel = 0;  // scratch is sized per representation
  d.sparse = true;
}

void DenseLMIConstraint::LoadDense(const std::vector<Entry>& lower, const double* C) {
  Storage& d = *data_;
  const size_t nn = Sq(n_);
  d.Aall.Reserve(nn * (m_ + 1));
  std::vector<std::vector<Entry>> by_var(m_);
  for (const Entry& e : lower) by_var[e.var].push_back(e);
  std::vector<double> M(nn);
  for (int i = 0; i < m_; i++) {
    std::fill(M.begin(), M.end(), 0.0);
    for (const Entry& e : by_var[i]) {
      M[static_cast<size_t>(e.c) * n_ + e.r] = e.val;
      M[static_cast<size_t>(e.r) * n_ + e.c] = e.val;
    }
    CudaCheck(cudaMemcpy(d.Aall.get() + nn * i, M.data(), sizeof(double) * nn, cudaMemcpyHostToDevice),
              "upload of an LMI matrix");
  }
  CudaCheck(cudaMemcpy(d.Aall.get() + nn * m_, C, sizeof(double) * nn, cudaMemcpyHostToDevice),
            "upload of LMI affine term");
  if (d.sparse) d.panel = 0;
  d.sparse = false;
}

// ---- HermitianPsdConstraint<Real> ------------------------------------------------------------------
HermitianPsdConstraint::HermitianPsdConstraint(int n, int m)
    : DenseLMIConstraint(n, m, EntrySparse{}), host_(std::make_shared<Host>()) {
  host_->entries.resize(m);
  host_->C.assign(Sq(n), 0.0);
  set_hermitian_semantics(true);
}

DenseLMIConstraint* HermitianPsdConstraint::Synced() {
  if (host_->dirty) {
    const int n = order(), m = number_of_variables();
    std::vector<Entry> lower;
    double nnz_full = 0;
    for (int i = 0; i < m; i++) {
      for (const auto& kv : host_->entries[i]) {
        if (kv.second == 0.0) continue;
        const int c = static_cast<int>(kv.first / n), r = static_cast<int>(kv.first % n);
        lower.push_back({i, r, c, kv.second});
        nnz_full += (r == c) ? 1 : 2;
      }
    }
    // Entry-sparse kernels do (sum nnz)^2 gathers, the dense path 1.33 m n^3 + 0.54 m^2 n^2 flops at
    // tensor-core rate: switch when the sparse count is clearly smaller.
    const double dense_work = 1.33 * m * static_cast<double>(n) * n * n + 0.54 * m * static_cast<double>(m) * n * n;
    if (nnz_full * nnz_full * 16.0 < dense_work) {
      LoadEntries(lower, host_->C.data());
    } else {
      LoadDense(lower, host_->C.data());
    }
    host_->dirty = false;
  }
  return this;
}

bool UpdateLinearOperator(HermitianPsdConstraint* o, double val, int var, int r, int c, int dim) {
  const int n = o->order();
  CONEX_DEMAND(dim < 1, "Complex dimension out of bounds.");
  CONEX_DEMAND(r < n && c < n, "Matrix dimension out of bounds.");
  CONEX_DEMAND((var >= 0) && (r >= 0) && (c >= 0), "Indices cannot be negative.");
  CONEX_DEMAND(var < o->number_of_variables(), "Variable index out of bounds.");
  const int hi = std::max(r, c), lo = std::min(r, c);
  o->host_->entries[var][static_cast<long>(lo) * n + hi] = val;
  o->host_->dirty = true;
  return false;
}

bool UpdateAffineTerm(HermitianPsdConstraint* o, double val, int r, int c, int dim) {
  const int n = o->order();
  CONEX_DEMAND(dim < 1, "Complex dimension out of bounds.");
  CONEX_DEMAND(r < n && c < n, "Matrix dimension out of bounds.");
  CONEX_DEMAND((r >= 0) && (c >= 0), "Indices cannot be negative.");
  o->host_->C[static_cast<size_t>(c) * n + r] = val;
  o->host_->C[static_cast<size_t>(r) * n + c] = val;
  o->host_->dirty = true;
  return false;
}

void DenseLMIConstraint::EnsureScratch() {
  Storage& d = *data_;
  if (d.panel != 0) return;
  const size_t nn = Sq(n_);
  if (d.sparse) {
    d.panel = 1;
    const size_t work = std::max(cxb_lanczos_worksize(n_), cxb_geodesic_worksize(n_));
    d.scratch.Resize(work);
    d.coef.Resize(m_ + 1);
    d.small.Resize(2 * (n_ / 2 + 2) + 8);
    d.iwork.Resize(2 * n_ + 8);
    d.rstart.Resize(n_);
    return;
  }
  // Modes: symmetric form (packed L^T A_i L, 0.54 A-sized second buffer; default when it fits), classic
  // form keeping every W A_i W (needed by the sharded exchange), or row panels through a bounded buffer.
  const size_t kp = cxb_packed_symmetric_size(n_);
  const size_t sym_bytes = sizeof(double) * (kp * (m_local_ + 2) + nn);
  const size_t full_bytes = sizeof(double) * nn * (m_local_ + 2);
  size_t free_bytes = 0, total_bytes = 0;
  CudaCheck(cudaMemGetInfo(&free_bytes, &total_bytes), "cudaMemGetInfo");
  const size_t other = sizeof(double) * (4 * nn + (size_t(1) << 28)) + (size_t(2) << 30);
  const int mode = ctx_->assembly_mode;
  bool sym_fits = sym_bytes + other <= free_bytes;
  bool full_fits = full_bytes + other <= free_bytes;
  if (sharded_) {
    // The form decides WHAT travels between the ranks (packed X with stride kp, or raw A with stride n^2)
    // and the size of the receive buffers, so it must be one decision for the whole communicator: a form
    // is used only if it fits on EVERY rank (shards differ by one matrix, free memory by whatever else
    // lives on each GPU). Both outcomes, including the failure below, are then identical on all ranks.
    int does_not_fit[2] = {sym_fits ? 0 : 1, full_fits ? 0 : 1};
    int* slot = ctx_->flags() + 6;
    CudaCheck(cudaMemcpyAsync(slot, does_not_fit, sizeof(does_not_fit), cudaMemcpyHostToDevice, ctx_->cuda_stream()),
              "H2D copy");
    Communicator::Get().AllReduceMaxInt(slot, 2, ctx_->cuda_stream());
    ctx_->DownloadInts(does_not_fit, slot, 2);
    sym_fits = does_not_fit[0] == 0;
    full_fits = does_not_fit[1] == 0;
  }
  d.symmetric = (mode == 3 || (mode == 0 && sym_fits)) && !(sharded_ && mode == 1);
  d.streamed = !sharded_ && !d.symmetric && (mode == 2 || ((mode == 0 || mode == 3) && !full_fits));
  if (sharded_ && !d.symmetric && !full_fits) {
    throw std::runtime_error("conex-b200: the scaled matrices of this shard do not fit in HBM; use more ranks");
  }
  // Constraint matrices scaled per pass. Streamed: a multiple of the 64-row GEMM tile, <= 2 GiB.
  const size_t budget = d.streamed ? (size_t(1) << 28) : (size_t(1) << 27);  // doubles
  size_t panel = std::max<size_t>(1, std::min<size_t>(m_local_ + 1, budget / nn));
  if (d.streamed && panel >= 64) panel -= panel % 64;
  d.panel = static_cast<int>(panel);
  d.T.Resize(nn * d.panel);
  if (d.symmetric) {
    d.X.Resize(kp * (m_local_ + 2));
    d.Lw.Resize(nn);
    // K2 on the integer tensor cores needs 8 bytes of slices per packed entry (as much as X); where they do not fit
    // beside everything else, K2 stays on the DMMA Gram
    const size_t slice_bytes = cxb_schur_dense_lmi_sym_gram_workspace(n_, m_local_);
    if (slice_bytes > 0 && sym_bytes + slice_bytes + other <= free_bytes) d.slices.Resize(slice_bytes);
  } else {
    d.B.Resize(d.streamed ? nn * (d.panel + 1) : nn * (m_local_ + 2));
  }
  if (sharded_) {
    const long ldl = WorkspaceSchurComplement::AugLd(m_local_);
    d.Hloc.Resize(static_cast<size_t>(ldl) * (m_local_ + 1));
    CudaCheck(cudaMemset(d.Hloc.get(), 0, sizeof(double) * d.Hloc.size()), "memset");
    // Exchanged chunks: up to 4 GiB each, never more than the largest shard
    const int world = Communicator::Get().world();
    const int largest = (m_ + world - 1) / world;
    // (a multiple of the 64-wide GEMM tile so that the block contractions have no ragged columns)
    size_t chunk = std::min<size_t>(largest, (size_t(1) << 29) / nn);
    if (chunk >= 64) chunk -= chunk % 64;
    d.chunk = static_cast<int>(std::max<size_t>(1, chunk));
    for (auto& r : d.recv) r.Resize((d.symmetric ? kp : nn) * d.chunk);
    CudaCheck(cudaStreamCreateWithFlags(&d.comm_stream, cudaStreamNonBlocking), "cudaStreamCreate");
    for (auto& e : d.arrived) CudaCheck(cudaEventCreateWithFlags(&e, cudaEventDisableTiming), "event");
    for (auto& e : d.consumed) CudaCheck(cudaEventCreateWithFlags(&e, cudaEventDisableTiming), "event");
    CudaCheck(cudaEventCreateWithFlags(&d.start, cudaEventDisableTiming), "event");
    if (d.symmetric && ctx_->peer_memory_exchange) ExchangePeerHandles();
  }
  const size_t work = std::max(cxb_lanczos_worksize(n_), cxb_geodesic_worksize(n_));
  d.scratch.Resize(work);
  d.coef.Resize(m_ + 1);
  d.small.Resize(2 * (n_ / 2 + 2) + 8);
  d.iwork.Resize(2 * n_ + 8);
  d.rstart.Resize(n_);
}

// Every rank publishes the CUDA IPC handle of its X buffer (64 bytes as 32 sixteen-bit words + an "ok" word, combined
// by an integer max all-reduce against zeros) and maps the others'. Any failure on any rank (IPC not permitted, no peer
// access) leaves ipc_ready false on ALL ranks and the exchange stays on ncclSend / ncclRecv.
void DenseLMIConstraint::ExchangePeerHandles() {
  Storage& d = *data_;
  Communicator& comm = Communicator::Get();
  const int world = comm.world(), rank = comm.rank();
  constexpr int kWords = 33;
  std::vector<int> words(static_cast<size_t>(world) * kWords + 1, 0);
  cudaIpcMemHandle_t mine;
  const bool have = cudaIpcGetMemHandle(&mine, d.X.get()) == cudaSuccess;
  if (!have) cudaGetLastError();
  if (have) {
    const unsigned char* bytes = reinterpret_cast<const unsigned char*>(&mine);
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handles are 64 bytes");
    int* slot = words.data() + static_cast<size_t>(rank) * kWords;
    slot[0] = 1;
    for (int i = 0; i < 32; i++) slot[1 + i] = bytes[2 * i] | (bytes[2 * i + 1] << 8);
  }
  d.ipc_words.Resize(words.size());
  cudaStream_t s = ctx_->cuda_stream();
  CudaCheck(cudaMemcpyAsync(d.ipc_words.get(), words.data(), sizeof(int) * words.size(), cudaMemcpyHostToDevice, s),
            "H2D copy");
  comm.AllReduceMaxInt(d.ipc_words.get(), words.size(), s);
  ctx_->DownloadInts(words.data(), d.ipc_words.get(), words.size());
  d.peer_x.assign(world, nullptr);
  int failed = 0;
  for (int p = 0; p < world; p++) {
    if (p == rank) continue;
    const int* slot = words.data() + static_cast<size_t>(p) * kWords;
    if (slot[0] != 1) {
      failed = 1;
      continue;
    }
    cudaIpcMemHandle_t h;
    unsigned char* bytes = reinterpret_cast<unsigned char*>(&h);
    for (int i = 0; i < 32; i++) {
      bytes[2 * i] = static_cast<unsigned char>(slot[1 + i] & 0xff);
      bytes[2 * i + 1] = static_cast<unsigned char>((slot[1 + i] >> 8) & 0xff);
    }
    void* mapped = nullptr;
    if (cudaIpcOpenMemHandle(&mapped, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
      cudaGetLastError();
      failed = 1;
      continue;
    }
    d.peer_x[p] = static_cast<double*>(mapped);
  }
  // one decision for the whole communicator
  int* flag = d.ipc_words.get() + words.size() - 1;
  CudaCheck(cudaMemcpyAsync(flag, &failed, sizeof(int), cudaMemcpyHostToDevice, s), "H2D copy");
  comm.AllReduceMaxInt(flag, 1, s);
  ctx_->DownloadInts(&failed, flag, 1);
  d.ipc_ready = failed == 0;
}

void SetIdentity(DenseLMIConstraint* o) {
  DeviceCheck(cxb_set_identity(o->ctx_->stream(), o->n_, o->workspace_.W.data), "cxb_set_identity");
}

void ConstructSchurComplementSystem(DenseLMIConstraint* o, bool initialize,
                                    SchurComplementSystem* sys) {
  // reference dense_lmi_constraint.cc:62-103; arithmetic described in device/schur.cu.
  o->EnsureScratch();
  auto& d = *o->data_;
  void* s = o->ctx_->stream();
  const int m = o->m_;
  if (!initialize) {
    throw std::runtime_error(
        "conex-b200: DenseLMIConstraint accumulates through the assembler (initialize == true)");
  }
  if (d.sparse) {
    DeviceCheck(cxb_sparse_lmi_schur(s, o->n_, m, d.sp_offsets.get(), d.sp_rows.get(), d.sp_cols.get(),
                                     d.sp_vals.get(), d.Cdense.get(), o->workspace_.W.data, d.sp_work.get(),
                                     sys->G.data, sys->G.ld),
                "cxb_sparse_lmi_schur");
  } else if (o->sharded_) {
    o->AssembleSharded(sys);
  } else if (d.symmetric) {
    int* flag = o->ctx_->flags() + 4;
    DeviceCheck(cxb_schur_dense_lmi_sym_scale(s, o->n_, m, d.Aall.get(), o->workspace_.W.data, d.X.get(), d.T.get(),
                                              d.panel, d.Lw.get(), flag),
                "cxb_schur_dense_lmi_sym_scale");
    DeviceCheck(cxb_schur_dense_lmi_sym_gram_ws(s, o->n_, m, d.X.get(), sys->G.data, sys->G.ld, d.slices.get(),
                                                d.slices.size()),
                "cxb_schur_dense_lmi_sym_gram_ws");
    int w_not_pd = 0;
    o->ctx_->DownloadInts(&w_not_pd, flag, 1);
    if (w_not_pd != 0) {
      // W lost numerical positive definiteness: the classic form does not need its Cholesky factor
      if (d.B.size() == 0) d.B.Resize(Sq(o->n_) * (o->m_local_ + 2));
      DeviceCheck(cxb_schur_dense_lmi(s, o->n_, m, d.Aall.get(), o->workspace_.W.data, d.B.get(), d.T.get(),
                                      d.panel, sys->G.data, sys->G.ld),
                  "cxb_schur_dense_lmi");
    }
  } else if (d.streamed) {
    DeviceCheck(cxb_schur_dense_lmi_streamed(s, o->n_, m, d.Aall.get(), o->workspace_.W.data, d.B.get(),
                                             d.T.get(), d.panel, sys->G.data, sys->G.ld),
                "cxb_schur_dense_lmi_streamed");
  } else
  DeviceCheck(cxb_schur_dense_lmi(s, o->n_, m, d.Aall.get(), o->workspace_.W.data, d.B.get(),
                                  d.T.get(), d.panel, sys->G.data, sys->G.ld),
              "cxb_schur_dense_lmi");
  const long ld = sys->G.ld;
  // rows m and m+1 of the augmented Gram hold AQc, <c,Qc> and AW, <w,c>.
  DeviceCheck(cxb_copy_strided(s, m, sys->G.data + m, ld, sys->AQc, 1), "cxb_copy_strided");
  DeviceCheck(cxb_copy_strided(s, m, sys->G.data + m + 1, ld, sys->AW, 1), "cxb_copy_strided");
  DeviceCheck(cxb_copy_strided(s, 1, sys->G.data + (long)m * ld + m + 1, 1, sys->scalars, 1),
              "cxb_copy_strided");
  DeviceCheck(cxb_copy_strided(s, 1, sys->G.data + (long)m * ld + m, 1, sys->scalars + 1, 1),
              "cxb_copy_strided");
}

// Sharded K1 + K2 (DESIGN.md "Multi-GPU"). Every rank
//   1. scales its own matrices and contracts its diagonal block with the single-GPU kernel chain
//      (cxb_schur_dense_lmi on the local m_local matrices; rows m_local, m_local+1 of the local
//      augmented Gram carry AQc_j, AW_j of the local j),
//   2. for each task of ShardPlan receives the peer's constraint matrices chunk by chunk
//      (ncclSend/ncclRecv on a side stream, double-buffered under the DMMA contraction) and
//      contracts them with its scaled matrices straight into the block's place in the global H,
//   3. sums the disjoint contributions with one ncclAllReduce over the augmented H — every entry
//      has exactly one non-zero contributor, so the sum is exact and H is bit-identical everywhere.
void DenseLMIConstraint::AssembleSharded(SchurComplementSystem* sys) {
  auto& d = *data_;
  Communicator& comm = Communicator::Get();
  cudaStream_t s = ctx_->cuda_stream();
  const int n = n_, m = m_, ml = m_local_, rb = row_begin_;
  const long nn = static_cast<long>(n) * n;
  const long ldg = sys->G.ld;
  const long ldl = WorkspaceSchurComplement::AugLd(ml);
  double* G = sys->G.data;
  // Symmetric form: every block of H is a product of packed scaled matrices X = L^T A L (W = L L^T,
  // factored redundantly and identically on every rank), and it is X that travels between ranks
  // (0.54 of the bytes of the raw matrices). Classic form: local W A_i W against the peers' raw A_j.
  const bool sym = d.symmetric;
  const long stride = sym ? static_cast<long>(cxb_packed_symmetric_size(n)) : nn;
  const double* local_scaled = sym ? d.X.get() : d.B.get();
  const double* send_source = sym ? d.X.get() : d.Aall.get();
  int* flag = ctx_->flags() + 4;

  for (auto& e : d.t_mark) {
    if (!e) CudaCheck(cudaEventCreate(&e), "cudaEventCreate");
  }
  CudaCheck(cudaEventRecord(d.t_mark[0], s), "cudaEventRecord");
  CudaCheck(cudaMemsetAsync(G, 0, sizeof(double) * ldg * (m + 1), s), "memset of H");

  // -- exchange schedule: a flat list of chunks over all distances --------------------------------
  struct Chunk {
    int from, recv_begin, recv_count;  // global indices of the matrices received (count 0: none)
    int to, send_begin, send_count;
    const PairTask* task;              // task the received chunk belongs to (nullptr: send only)
  };
  const std::vector<PairTask> plan = ShardPlan(m, comm.world(), comm.rank());
  std::vector<Chunk> chunks;
  for (int dist = 1; dist <= comm.world() / 2; dist++) {
    const PairTask* task = nullptr;
    for (const auto& t : plan) {
      if (t.peer == (comm.rank() + dist) % comm.world()) task = &t;
    }
    const SendTask snd = ShardSend(m, comm.world(), comm.rank(), dist);
    const int nrecv = task ? (task->col_count + d.chunk - 1) / d.chunk : 0;
    const int nsend = (snd.count + d.chunk - 1) / d.chunk;
    for (int c = 0; c < std::max(nrecv, nsend); c++) {
      Chunk ch{};
      ch.task = nullptr;
      if (c < nrecv) {
        ch.from = task->peer;
        ch.recv_begin = task->col_begin + c * d.chunk;
        ch.recv_count = std::min(d.chunk, task->col_begin + task->col_count - ch.recv_begin);
        ch.task = task;
      }
      if (c < nsend) {
        ch.to = snd.to;
        ch.send_begin = snd.begin + c * d.chunk;
        ch.send_count = std::min(d.chunk, snd.begin + snd.count - ch.send_begin);
      }
      chunks.push_back(ch);
    }
  }
  // Symmetric form with peer memory mapped: chunks are pulled from the peer's X by a copy engine over NVLink.
  const bool pull = sym && d.ipc_ready;
  auto post = [&](size_t c) {  // enqueue the transfer of chunk c on the side stream
    const Chunk& ch = chunks[c];
    const int buf = static_cast<int>(c % 2);
    if (c >= 2) CudaCheck(cudaStreamWaitEvent(d.comm_stream, d.consumed[buf], 0), "cudaStreamWaitEvent");
    if (pull) {
      if (ch.recv_count > 0) {
        const int peer_begin = ShardBegin(m, comm.world(), ch.from);
        CudaCheck(cudaMemcpyAsync(d.recv[buf].get(), d.peer_x[ch.from] + static_cast<long>(ch.recv_begin - peer_begin) * stride,
                                  sizeof(double) * static_cast<size_t>(ch.recv_count) * stride, cudaMemcpyDefault,
                                  d.comm_stream),
                  "peer copy of a chunk of scaled matrices");
      }
    } else {
      const double* src = ch.send_count ? send_source + static_cast<long>(ch.send_begin - rb) * stride : nullptr;
      comm.SendRecv(src, static_cast<size_t>(ch.send_count) * stride, ch.to, d.recv[buf].get(),
                    static_cast<size_t>(ch.recv_count) * stride, ch.from, d.comm_stream);
    }
    CudaCheck(cudaEventRecord(d.arrived[buf], d.comm_stream), "cudaEventRecord");
  };
  auto release_side_stream = [&]() {
    CudaCheck(cudaEventRecord(d.start, s), "cudaEventRecord");
    CudaCheck(cudaStreamWaitEvent(d.comm_stream, d.start, 0), "cudaStreamWaitEvent");
    // every rank's X must be complete before anyone pulls from it: a one-word all-reduce on the side streams is that
    // barrier (each rank enqueues it behind its own K1)
    if (pull) comm.AllReduceMaxInt(d.ipc_words.get(), 1, d.comm_stream);
    if (!chunks.empty()) post(0);
  };
  // Classic form: the raw matrices can travel while the local block is computed. Symmetric form: the
  // scaled matrices exist only after the local K1, so the first transfer starts after the local block.
  if (!sym) release_side_stream();

  // -- 1. local diagonal block ----------------------------------------------------------------------
  if (sym) {
    // K1 first; the scaled matrices can travel from here on, under the local Gram
    DeviceCheck(cxb_schur_dense_lmi_sym_scale(s, n, ml, d.Aall.get(), workspace_.W.data, d.X.get(), d.T.get(), d.panel,
                                              d.Lw.get(), flag),
                "cxb_schur_dense_lmi_sym_scale(local block)");
    release_side_stream();
    DeviceCheck(cxb_schur_dense_lmi_sym_gram_ws(s, n, ml, d.X.get(), d.Hloc.get(), ldl, d.slices.get(), d.slices.size()),
                "cxb_schur_dense_lmi_sym_gram_ws(local block)");
  } else {
    DeviceCheck(cxb_schur_dense_lmi(s, n, ml, d.Aall.get(), workspace_.W.data, d.B.get(), d.T.get(),
                                    d.panel, d.Hloc.get(), ldl),
                "cxb_schur_dense_lmi(local block)");
  }
  // H[rb.., rb..] <- Hloc[0:ml, 0:ml]; rows m, m+1 (AQc, AW) <- rows ml, ml+1 of the local columns
  CudaCheck(cudaMemcpy2DAsync(G + static_cast<long>(rb) * ldg + rb, sizeof(double) * ldg, d.Hloc.get(),
                              sizeof(double) * ldl, sizeof(double) * ml, ml, cudaMemcpyDeviceToDevice, s),
            "copy of the diagonal block");
  CudaCheck(cudaMemcpy2DAsync(G + static_cast<long>(rb) * ldg + m, sizeof(double) * ldg,
                              d.Hloc.get() + ml, sizeof(double) * ldl, sizeof(double) * 2, ml,
                              cudaMemcpyDeviceToDevice, s),
            "copy of the residual rows");
  if (comm.rank() == 0) {  // <c,Qc> and <w,c> are the same on every rank: contributed once
    CudaCheck(cudaMemcpyAsync(G + static_cast<long>(m) * ldg + m, d.Hloc.get() + static_cast<long>(ml) * ldl + ml,
                              sizeof(double) * 2, cudaMemcpyDeviceToDevice, s),
              "copy of the scalars");
  }

  CudaCheck(cudaEventRecord(d.t_mark[1], s), "cudaEventRecord");
  while (d.t_chunk.size() < 3 * chunks.size()) {
    cudaEvent_t e = nullptr;
    CudaCheck(cudaEventCreate(&e), "cudaEventCreate");
    d.t_chunk.push_back(e);
  }
  d.t_chunks_used = chunks.size();

  // -- 2. off-diagonal blocks ----------------------------------------------------------------------
  for (size_t c = 0; c < chunks.size(); c++) {
    if (c + 1 < chunks.size()) post(c + 1);
    const Chunk& ch = chunks[c];
    const int buf = static_cast<int>(c % 2);
    CudaCheck(cudaEventRecord(d.t_chunk[3 * c], s), "cudaEventRecord");
    CudaCheck(cudaStreamWaitEvent(s, d.arrived[buf], 0), "cudaStreamWaitEvent");
    CudaCheck(cudaEventRecord(d.t_chunk[3 * c + 1], s), "cudaEventRecord");
    if (ch.recv_count > 0) {
      const PairTask& t = *ch.task;
      const double* Bl = local_scaled + static_cast<long>(t.row_begin - rb) * stride;
      if (t.peer < comm.rank()) {
        // block below the diagonal: H[rows, cols] = <scaled rows, received cols>
        DeviceCheck(cxb_dgemm(s, 1, 0, t.row_count, ch.recv_count, static_cast<int>(stride), 1.0, Bl, stride, 0,
                              d.recv[buf].get(), stride, 0, 0.0,
                              G + static_cast<long>(ch.recv_begin) * ldg + t.row_begin, ldg, 0, 1, 0),
                    "cxb_dgemm(off-diagonal block)");
      } else {
        // block above the diagonal: store its transpose H[cols, rows]
        DeviceCheck(cxb_dgemm(s, 1, 0, ch.recv_count, t.row_count, static_cast<int>(stride), 1.0,
                              d.recv[buf].get(), stride, 0, Bl, stride, 0, 0.0,
                              G + static_cast<long>(t.row_begin) * ldg + ch.recv_begin, ldg, 0, 1, 0),
                    "cxb_dgemm(off-diagonal block, transposed)");
      }
    }
    CudaCheck(cudaEventRecord(d.consumed[buf], s), "cudaEventRecord");
    CudaCheck(cudaEventRecord(d.t_chunk[3 * c + 2], s), "cudaEventRecord");
  }
  // -- 3. one all-reduce over the augmented H -------------------------------------------------------
  CudaCheck(cudaEventRecord(d.t_mark[2], s), "cudaEventRecord");
  comm.AllReduceSum(G, static_cast<size_t>(ldg) * (m + 1), s);
  CudaCheck(cudaEventRecord(d.t_mark[3], s), "cudaEventRecord");
  if (sym) {
    // W is replicated bit-identically, so every rank sees the same flag and takes the same branch.
    int w_not_pd = 0;
    ctx_->DownloadInts(&w_not_pd, flag, 1);
    if (w_not_pd != 0) {
      d.symmetric = false;
      if (d.B.size() == 0) d.B.Resize(Sq(n) * (ml + 2));
      for (auto& r : d.recv) r.Reserve(static_cast<size_t>(nn) * d.chunk);
      AssembleSharded(sys);
    }
  }
}

void DenseLMIConstraint::ComputeNegativeSlack(double k, const Ref& y, Ref* minus_s) {
  auto& d = *data_;
  if (d.sparse) {
    DeviceCheck(cxb_sparse_lmi_slack(ctx_->stream(), n_, d.npos, d.sp_pos_ptr.get(), d.sp_pos_index.get(),
                                     d.sp_pos_var.get(), d.sp_pos_val.get(), d.Cdense.get(), y.data, k,
                                     minus_s->data),
                "cxb_sparse_lmi_slack");
    return;
  }
  ctx_->CopyOnDevice(d.coef.get(), y.data + row_begin_, m_local_);
  // the affine term is added once (rank 0); the other ranks contribute 0 * C
  const double c_coef = (!sharded_ || Communicator::Get().rank() == 0) ? -k : 0.0;
  DeviceCheck(cxb_fill(ctx_->stream(), 1, c_coef, d.coef.get() + m_local_), "cxb_fill");
  DeviceCheck(cxb_gemv_n(ctx_->stream(), (long)Sq(n_), m_local_ + 1, d.Aall.get(), d.coef.get(),
                         minus_s->data),
              "cxb_gemv_n");
  if (sharded_) Communicator::Get().AllReduceSum(minus_s->data, Sq(n_), ctx_->cuda_stream());
}

DenseLMIConstraint::SpectrumEstimate DenseLMIConstraint::EstimateSpectrum(const Ref& WS,
                                                                          const Ref& start_matrix) {
  // reference psd_constraint.cc:63-80 / :107-127 and approximate_eigenvalues.cc:241-256.
  auto& d = *data_;
  void* s = ctx_->stream();
  const int n = n_;
  const int num_iter = hermitian_ ? n / 2 + 1 : n / 2;
  const int cap = n / 2 + 2;
  double* alpha = d.small.get();
  double* beta = alpha + cap;
  double* red = beta + cap;  // 8 slots
  int* count = d.iwork.get() + 2 * n + 2;  // two ints: step count, stop flag
  DeviceCheck(cxb_ws_reductions(s, n, WS.data, red), "cxb_ws_reductions");
  if (hermitian_) {
    // T::Random(n, 1) = Eigen::MatrixXd::Random: n draws of -1 + 2 rand() / RAND_MAX
    // (jordan_matrix_algebra.cc:81-87); drawn even for n == 1 so the libc stream stays aligned.
    double* r = ctx_->pinned().get();
    if (static_cast<size_t>(n) > ctx_->pinned().size()) {
      ctx_->Synchronize();
      ctx_->pinned().Reserve(n);
      r = ctx_->pinned().get();
    }
    for (int i = 0; i < n; i++) r[i] = -1.0 + 2.0 * static_cast<double>(std::rand()) / static_cast<double>(RAND_MAX);
    ctx_->Upload(d.rstart.get(), r, n);
  }
  if (n > 1 && num_iter >= 1) {
    const double* start = hermitian_ ? d.rstart.get() : start_matrix.data;
    const double* column = hermitian_ ? nullptr : red + 2;
    const double rel_tol = hermitian_ ? 1e-5 : 0.0;
    // Long recurrences usually break down early (beta^2 below the threshold): run a short first range,
    // look at the stop flag, and launch the rest only when needed.
    constexpr int kProbe = 32;
    int first_end = num_iter;
    if (num_iter > 4 * kProbe) first_end = kProbe;
    DeviceCheck(cxb_lanczos_two_sided_range(s, n, WS.data, workspace_.W.data, start, column, num_iter, 0, first_end,
                                            alpha, beta, count, d.scratch.get(), rel_tol),
                "cxb_lanczos_two_sided_range");
    if (first_end < num_iter) {
      int state[2] = {0, 0};
      ctx_->DownloadInts(state, count, 2);
      if (state[1] == 0) {
        DeviceCheck(cxb_lanczos_two_sided_range(s, n, WS.data, workspace_.W.data, start, column, num_iter, first_end,
                                                num_iter, alpha, beta, count, d.scratch.get(), rel_tol),
                    "cxb_lanczos_two_sided_range");
      }
    }
  }
  std::vector<double> host(2 * cap + 8);
  int cnt = 0;
  CudaCheck(cudaMemcpyAsync(host.data(), d.small.get(), sizeof(double) * host.size(),
                            cudaMemcpyDeviceToHost, ctx_->cuda_stream()),
            "D2H Lanczos coefficients");
  if (n > 1) {
    ctx_->DownloadInts(&cnt, count, 1);
  } else {
    ctx_->Synchronize();
  }
  static const bool trace = std::getenv("CONEX_TRACE_EIGEN") != nullptr;
  if (trace) std::cerr << "[conex-b200 trace] Lanczos steps " << cnt + 1 << " of " << num_iter << std::endl;
  SpectrumEstimate e;
  e.trace = host[2 * cap + 0];
  e.trace_of_square = host[2 * cap + 1];
  if (n == 1) {
    e.ritz_min = e.ritz_max = e.trace;  // ApproximateEigenvalues returns WS itself for n == 1
  } else {
    std::vector<double> a(host.begin(), host.begin() + cnt + 1);
    std::vector<double> b(host.begin() + cap, host.begin() + cap + cnt);
    const auto mm = ExtremeEigenvaluesOfTridiagonal(a, b);
    e.ritz_min = mm.first;
    e.ritz_max = mm.second;
  }
  return e;
}

void PrepareStep(DenseLMIConstraint* o, const StepOptions& opt, const Ref& y, StepInfo* info) {
  // reference psd_constraint.cc:45-84. There minus_s and WS alias temp_1; here minus_s lives in
  // temp_1 and WS in temp_2 (WSWS is never formed: tr(WS WS) is an O(n^2) reduction).
  auto& w = o->workspace_;
  void* s = o->ctx_->stream();
  const int n = o->n_;
  Ref minus_s = w.temp_1, WS = w.temp_2;
  o->EnsureScratch();
  o->ComputeNegativeSlack(opt.c_weight, y, &minus_s);
  DeviceCheck(cxb_dgemm(s, 0, 0, n, n, n, 1.0, w.W.data, n, 0, minus_s.data, n, 0, 0.0, WS.data, n, 0,
                        1, 0),
              "cxb_dgemm(W*S)");
  if (opt.affine) {
    // AffineUpdate (psd_constraint.cc:33-43): W <- (1 + e) W + (WS) W
    DeviceCheck(cxb_dgemm(s, 0, 0, n, n, n, 1.0, WS.data, n, 0, w.W.data, n, 0, 0.0, minus_s.data, n,
                          0, 1, 0),
                "cxb_dgemm(WS*W)");
    DeviceCheck(cxb_affine_update(s, n, w.W.data, minus_s.data, opt.e_weight), "cxb_affine_update");
    return;
  }
  // The reference starts Lanczos from minus_s.col(argmax diag WS) *after* WS overwrote minus_s,
  // i.e. from a column of WS (psd_constraint.cc:48-50,66-69).
  const auto e = o->EstimateSpectrum(WS, WS);
  const double lambda_1 = std::fabs(opt.e_weight + e.ritz_min);
  const double lambda_2 = std::fabs(opt.e_weight + e.ritz_max);
  info->norminfd = std::max(lambda_1, lambda_2);
  info->normsqrd = e.trace_of_square + 2 * e.trace + n;
}

bool TakeStep(DenseLMIConstraint* o, const StepOptions& opt) {
  // reference psd_constraint.cc:86-90 -> GeodesicUpdate :13-28
  auto& d = *o->data_;
  auto& w = o->workspace_;
  if (o->hermitian_) {
    DeviceCheck(cxb_geodesic_update_taylor(o->ctx_->stream(), o->n_, w.W.data, w.temp_2.data, opt.e_weight,
                                           opt.step_size, d.scratch.get()),
                "cxb_geodesic_update_taylor");
    return true;
  }
  DeviceCheck(cxb_geodesic_update(o->ctx_->stream(), o->n_, w.W.data, w.temp_2.data, opt.e_weight,
                                  opt.step_size, d.scratch.get(), d.iwork.get(),
                                  d.iwork.get() + 2 * o->n_ + 1),
              "cxb_geodesic_update");
  return true;
}

void GetWeightedSlackEigenvalues(DenseLMIConstraint* o, const Ref& y, double c_weight,
                                 WeightedSlackEigenvalues* p) {
  // reference psd_constraint.cc:97-128: here the start vector is a column of the true -S.
  auto& w = o->workspace_;
  void* s = o->ctx_->stream();
  const int n = o->n_;
  Ref minus_s = w.temp_1, WS = w.temp_2;
  o->EnsureScratch();
  static const bool trace = std::getenv("CONEX_TRACE_EIGEN") != nullptr;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  if (trace) {
    for (auto& e : ev) cudaEventCreate(&e);
    cudaEventRecord(ev[0], o->ctx_->cuda_stream());
  }
  o->ComputeNegativeSlack(c_weight, y, &minus_s);
  if (trace) cudaEventRecord(ev[1], o->ctx_->cuda_stream());
  DeviceCheck(cxb_dgemm(s, 0, 0, n, n, n, 1.0, w.W.data, n, 0, minus_s.data, n, 0, 0.0, WS.data, n, 0,
                        1, 0),
              "cxb_dgemm(W*S)");
  if (trace) cudaEventRecord(ev[2], o->ctx_->cuda_stream());
  const auto t0 = std::chrono::high_resolution_clock::now();
  const auto e = o->EstimateSpectrum(WS, minus_s);
  if (trace) {
    const double host_ms =
        std::chrono::duration<double, std::milli>(std::chrono::high_resolution_clock::now() - t0).count();
    cudaEventRecord(ev[3], o->ctx_->cuda_stream());
    cudaEventSynchronize(ev[3]);
    float a = 0, b = 0;
    cudaEventElapsedTime(&a, ev[0], ev[1]);
    cudaEventElapsedTime(&b, ev[1], ev[2]);
    std::cerr << "[conex-b200 trace] eigen-bound: slack " << a << " ms, W*S " << b << " ms, spectrum (host wall) "
              << host_ms << " ms" << std::endl;
    for (auto& x : ev) cudaEventDestroy(x);
  }
  p->lambda_max = -e.ritz_min;
  p->lambda_min = -e.ritz_max;
  p->frobenius_norm_squared = e.trace_of_square;
  p->trace = -e.trace;
}

}  // namespace conex

/* conex-b200 extensions to the conex C ABI (include/conex.h).
 *
 * None of these exist in the reference; they expose what its C++ tests reach through the headers under conex/
 * (GetFeasibleObjective, Program::Status, the REPORT() stream) plus device-resident construction
 * and timing hooks needed to benchmark on the GPU. All take the opaque program handle returned by
 * CONEX_CreateConeProgram. Host pointers unless a parameter is named d_*.
 */
#ifndef CONEX_B200_H
#define CONEX_B200_H
#include "conex.h"
#ifdef __cplusplus
extern "C" {
#endif

/* b = AW/2 at W = I (reference GetFeasibleObjective, cone_program.cc:535-545). Writes m doubles. */
void CONEXB200_FeasibleObjective(void* prog, double* b);

/* out4 = {solved, num_iterations, primal_infeasible, dual_infeasible} (Program::Status()). */
void CONEXB200_GetStatus(void* prog, int* out4);

/* out8 = {inv_sqrt_mu, mu, d_2, d_inf, by, cx, kkt_error, step_size} of iteration `iter` of the
 * last solve — the values the reference REPORT()s to stdout (cone_program.cc:456-468).
 * Returns 1, or 0 when `iter` is out of range. */
int CONEXB200_GetIterationLog(void* prog, int iter, double* out8);

/* The three terms the logged cx of iteration `iter` (negative: from the end) is formed from (reference
 * cone_program.cc:447-452):  k b_s cx = out3[0] + out3[1] - out3[2] = 2 <c,w> + <AQc, y> - k c_s <c,Qc>. Late in a solve
 * the last two are ~k^2 times larger than their difference: (|out3[0]| + |out3[1]| + |out3[2]|) / |their sum| is the
 * condition number of that formula, i.e. what the rounding errors of the inner products are amplified by in cx. */
int CONEXB200_GetObjectiveTerms(void* prog, int iter, double* out3);

/* Device time (ms, CUDA events on the program's stream) of Newton step `iter` of the last solve;
 * returns 0 when out of range. */
int CONEXB200_GetIterationMilliseconds(void* prog, int iter, double* ms);

/* Device milliseconds of the five phases of Newton step `iter`: out5 = {assemble, factor, mu, solve,
 * update} (CUDA events at the phase boundaries, cone_program.cc:338-437 in the reference). */
int CONEXB200_GetIterationPhaseMilliseconds(void* prog, int iter, double* out5);

/* Wall-clock seconds per phase {assemble, factor, solve, update, mu} of the last solve, the five
 * phases the reference wraps in START_TIMER (cone_program.cc:338-437). Summed from the per-iteration
 * CUDA events; CONEXB200_SetTiming is kept for ABI stability and has no effect. */
void CONEXB200_SetTiming(void* prog, int enabled);
void CONEXB200_GetPhaseSeconds(void* prog, double* out5);

/* Assembles the Newton system at the current iterate (coldstart != 0: at W = I) and copies it to
 * host memory: H (m x m column-major, lower triangle valid), AW, AQc (m), scalars2 = {<w,c>, <c,Qc>}. */
void CONEXB200_AssembleNewtonSystem(void* prog, int coldstart, double* H, double* AW, double* AQc,
                                    double* scalars2);

/* CONEX_AddDenseLMIConstraint with the matrices already in device memory (d_A: m contiguous
 * column-major n x n blocks, d_C: n x n). The data is copied device-to-device. */
int CONEXB200_AddDenseLMIConstraintDevice(void* prog, const double* d_A, int n, int m,
                                          const double* d_C);

/* ---- multi-GPU: one process per GPU, NCCL over NVLink 5 / NVSwitch (DESIGN.md "Multi-GPU") ----------
 * Rendezvous: rank 0 calls CONEXB200_CommGetUniqueId and ships the 128 bytes to the other ranks by
 * any means (torch.distributed, MPI, a file); every rank then calls CONEXB200_CommInitRank after
 * selecting its device (cudaSetDevice / torch.cuda.set_device). All return 0 on success, 1 on failure
 * (message on stderr). With world == 1 no NCCL is needed and none is loaded. */
int CONEXB200_CommGetUniqueId(char* out128);
int CONEXB200_CommInitRank(int world, int rank, const char* id128);
void CONEXB200_CommDestroy(void);
int CONEXB200_CommWorld(void);
int CONEXB200_CommRank(void);

/* The 1-D row partition used for a sharded block: rank r owns the constraint matrices
 * [begin, begin + count) of m. */
void CONEXB200_ShardRange(int m, int world, int rank, int* begin, int* count);
/* The off-diagonal block tasks of `rank` (host logic, no GPU): writes up to `capacity` records of
 * five ints {peer, row_begin, row_count, col_begin, col_count} and returns the number of tasks. */
int CONEXB200_ShardPlan(int m, int world, int rank, int* out5, int capacity);

/* This rank's shard of a dense LMI block with m constraint matrices in total: d_A_local holds the
 * rank's own matrices (CONEXB200_ShardRange) as contiguous column-major n x n blocks in device
 * memory, d_C the full affine term. Every rank of the communicator must add the same block. The
 * solve calls (CONEX_Maximize, ...) are then collective: every rank calls them with the same
 * arguments and receives the same y. */
int CONEXB200_AddDenseLMIConstraintShard(void* prog, const double* d_A_local, int n, int m,
                                         const double* d_C);

/* Marks a program that is NOT sharded as collective: every rank of the communicator has built the
 * same program (same data, same call sequence) and calls its solves in lock step, so that the
 * replicated phases with enough flops may be split across the ranks — today the Cholesky of the
 * Schur complement (below). Programs holding a sharded block are collective by construction. */
void CONEXB200_SetCollective(void* prog, int collective);

/* Multi-GPU Cholesky of collective programs (reference: BlockCholeskyInPlace on one thread,
 * block_triangular_operations.cc:184-219): block columns of `block` columns (<= 512) dealt 1-D
 * block-cyclically to the ranks, each factored panel broadcast over NCCL with a look-ahead of one
 * panel, trailing updates on the owners; every rank ends with the complete factor. Used when the
 * KKT order is >= min_order (default 4096; smaller systems are factored replicated). Process-wide;
 * a negative min_order / non-positive block leaves that setting unchanged. */
void CONEXB200_SetDistributedCholesky(int min_order, int block);
/* Host logic of that schedule (no GPU): writes up to `capacity` records {kind, panel, target} of the
 * operations `rank` enqueues — kind 0 factor `panel`, 1 broadcast `panel` from rank `target`, 2 wait
 * for `panel`, 3 update block column `target` with `panel` — and returns their number. */
int CONEXB200_CholeskySchedule(int N, int block, int world, int rank, int* out3, int capacity);
/* The distributed factorisation alone, collective: d_H (N x N, lower, leading dimension ld, device)
 * must hold the same matrix on every rank and is overwritten by the complete factor on every rank.
 * *info = 0, or non-zero on every rank if the matrix is not positive definite. Returns 0 / 1. */
int CONEXB200_DistributedPotrf(int N, double* d_H, long ld, int block, int* info);

/* Sharded LMI blocks (symmetric form) exchange their packed scaled matrices through PEER MEMORY by default: every rank
 * maps the others' buffers (CUDA IPC) and pulls its chunks with copy engines over NVLink, behind a one-word all-reduce
 * that says everyone's matrices are complete; 0 = always ncclSend / ncclRecv (also the automatic fallback when IPC
 * mapping fails on any rank). Call before the first solve, with the same value on every rank. */
void CONEXB200_SetPeerMemoryExchange(void* prog, int enabled);

/* Where the last sharded assembly of LMI constraint `id` spent its device time on THIS rank (CUDA events on the
 * compute stream): out4 = {local K1 + diagonal block, stalls waiting for a peer's chunk (exchange not hidden),
 * off-diagonal contractions, all-reduce of H} in ms. Returns 1, or 0 when the constraint is not sharded. */
int CONEXB200_GetShardPhaseMilliseconds(void* prog, int id, double* out4);

/* Zero-copy variant for operators that only fit once: the library allocates this rank's storage
 * (local_count = CONEXB200_ShardRange(m, world, rank) matrices, then C) and returns device pointers
 * that the caller fills in place (column-major n x n blocks) before the first solve. With world == 1
 * this is the whole block. Returns the constraint id, or -1. */
int CONEXB200_NewDenseLMIConstraintStorage(void* prog, int n, int m, double** d_A_local, double** d_C);

/* Schur assembly of LMI blocks of `prog`: 0 = decide from free HBM (default: symmetric form when it
 * fits, else row panels), 1 = classic form keeping all W A_i W (a second A-sized buffer; one Gram GEMM),
 * 2 = stream row panels (A + 2 panels), 3 = symmetric form: packed L^T A_i L with W = L L^T and a
 * SYRK-shaped Gram (0.54 A-sized buffer, 2.2x fewer flops). Call before the first solve. Same H in
 * every mode up to rounding (different summation order). */
void CONEXB200_SetAssemblyMode(void* prog, int mode);

/* Host-logic probes that need no GPU: the closed-form mu rule (reference divergence.cc:96-111) and
 * the extreme eigenvalues of a Lanczos Jacobi matrix (alpha: n, beta: n-1; out2 = {min, max}). */
double CONEXB200_DivergenceUpperBoundInverse(double bound, double frobenius_norm_squared,
                                             double trace, double lambda_min, double lambda_max,
                                             double rank);
void CONEXB200_TridiagonalExtremes(int n, const double* alpha, const double* beta, double* out2);

/* Number of CUDA kernels launched by this library in the current process so far. */
long CONEXB200_LaunchCount();

/* 1 when a CUDA device of compute capability 10.x is usable, else 0 (the library has no CPU path:
 * solves then fail with a message on stderr). */
int CONEXB200_DeviceAvailable();

/* ---- cones the reference builds through C++ constructors only -------------------------------- */
/* SOCConstraint(A, c) (conex/soc_constraint.h:9-15): c - A y in the Lorentz cone of R^{n+1};
 * A is (n + 1) x m column-major. Returns the constraint id. */
int CONEXB200_AddSocConstraint(void* prog, int n, int m, const double* A, const double* c);
/* The LP cone and the second-order cone on a list of `nvars` distinct variables `vars`, like
 * CONEX_AddSparseLMIConstraint for LMIs (Program::AddConstraint(cone, variables)):
 *   CONEXB200_AddSparseLinearConstraint: c - A y[vars] >= 0, A rows x nvars column-major, c `rows` entries;
 *   CONEXB200_AddSparseSocConstraint:    c - A y[vars] in the Lorentz cone of R^{n+1}, A (n + 1) x nvars.
 * The program's number of variables must be set. Duplicate or out-of-range variables add nothing and return -1;
 * otherwise the constraint id. */
int CONEXB200_AddSparseLinearConstraint(void* prog, const double* A, int rows, int nvars, const double* c,
                                        const long* vars);
int CONEXB200_AddSparseSocConstraint(void* prog, int n, int nvars, const double* A, const double* c,
                                     const long* vars);
/* Program::AddConstraint(EqualityConstraints{A, b}[, vars]) (conex/cone_program.h:193-217):
 * A y[vars] = b, A rows x nvars column-major, vars == NULL means all variables. The multipliers
 * become extra unknowns of the KKT system, which is then factored by the regularised LDL^T. */
int CONEXB200_AddEqualityConstraint(void* prog, int rows, int nvars, const double* A, const double* b,
                                    const long* vars);
/* 1 when constraint `id` (an LMI built through CONEX_NewLinearMatrixInequality) is held in entry-sparse
 * form and assembled by gathers from W, 0 when it is dense, -1 for other constraint types. Valid after
 * the first solve. */
int CONEXB200_ConstraintIsEntrySparse(void* prog, int id);
/* The form in which LMI constraint `id` assembles its Schur complement (CONEXB200_SetAssemblyMode; decided at the
 * first assembly): 0 undecided, 1 classic, 2 row panels, 3 symmetric, 4 entry-sparse gathers; -1 for other cones. */
int CONEXB200_GetAssemblyForm(void* prog, int id);
/* ---- chordal-sparse programs: cones on overlapping subsets of the variables (reference
 * SupernodalKKTSolver, kkt_solver.h:16-65 + clique_ordering.cc + block_triangular_operations.cc) -----
 * kind 0 (default): decide from the cones' variable sets — the multifrontal solver
 * (host/supernodal_kkt_solver.h) when there is more than one supernode, at least 256 unknowns and it
 * saves at least half of the dense factorisation's flops; 1: always one dense supernode; 2: always
 * multifrontal (fails for programs with equality multipliers or collective programs). Call before
 * the first solve. */
void CONEXB200_SetKKTSolverKind(void* prog, int kind);
/* Supernodes of the KKT solver in use (1 = dense); valid after the first solve / assembly. */
int CONEXB200_GetNumberOfSupernodes(void* prog);
/* Host logic of the symbolic step (no GPU). Cliques in CSR form (clique_ptr: num_cliques + 1 entries).
 * Outputs: position[v] = place of variable v in the elimination order, node_of[v] = supernode that
 * eliminates it, supernodes and separators in CSR form (node_ptr / sep_ptr: nodes + 1 entries; at most
 * N nodes; node_vars: N entries; sep_vars: sep_capacity entries), flops2 = {multifrontal, dense N^3/3}.
 * Returns the number of supernodes, -(needed sep_capacity) if sep_vars is too small, -1 on bad input. */
int CONEXB200_SupernodalAnalysis(int N, int num_cliques, const int* clique_ptr, const int* clique_vars,
                                 int* position, int* node_of, int* node_ptr, int* node_vars, int* sep_ptr,
                                 int* sep_vars, int sep_capacity, double* flops2);
/* A new program on the memory of `other` (reference `Program prog2(m, &prog.memory_)`, cone_program.h:106-109,
 * test_warmstart.cc:47-79): after adding the same constraints in the same order, a solve with
 * initialization_mode = warm start continues from `other`'s iterate (scaling points and scalings live in that
 * memory). `other` must outlive the new program and the two must not solve concurrently. NULL on failure. */
void* CONEXB200_CreateConeProgramOnMemoryOf(void* other);
/* Constraints added so far (Program::NumberOfConstraints, conex/cone_program.h); CONEX_AddLinearInequalities adds
 * zero, one or two (an LP cone for the finite bounds, an equality block for rows with lb == ub). */
int CONEXB200_NumberOfConstraints(void* prog);
/* Variables + equality multipliers (conex/constraint_manager.h:42-48). */
int CONEXB200_SizeOfKKTSystem(void* prog);
/* Host-logic probe: the pivot order Eigen::RLDLT derives from the diagonal (RLDLT.h:328-356). */
void CONEXB200_RldltPivotOrder(int n, const double* diag, int* perm);

/* ---- many small programs in lock step (BASELINE config 3) ------------------------------------
 * `programs`: `count` handles built through the CONEX_* calls with identical structure (same number
 * of variables, same list of LP / second-order / dense-LMI cones, each on the same list of distinct
 * variables in every program — all of them, or any subset in any order, as CONEX_AddSparseLMIConstraint,
 * CONEXB200_AddSparseLinearConstraint and CONEXB200_AddSparseSocConstraint build them — and the same
 * equality blocks — rows, variable subset, position among the cones — e.g. the lb == ub rows of
 * CONEX_AddLinearInequalities; at least one cone). A variable that no cone covers leaves the KKT
 * system singular, as in CONEX_Maximize. CONEXB200_CreateBatch packs their data into
 * batched device arrays (the handles may be deleted afterwards); it returns NULL for mismatched
 * structures. CONEXB200_BatchMaximize solves all of them: b and y are m x count column-major HOST
 * arrays, solved[p] / the return value follow CONEX_Maximize (1 = solved; the return value is the
 * number of solved programs, -1 on an error). Every program follows the same iteration sequence it
 * would follow through CONEX_Maximize alone, from a cold start or, with initialization_mode = 1, warm-
 * started from the iterate of the batch's previous solve (-1 when there was none). With equality
 * blocks the KKT systems are factored by a batched regularised LDL^T; iterative_refinement_iterations
 * > 0 is then refused (-1), as is enable_line_search when every constraint is an LP cone or an
 * equality block. The KKT order N (variables + multipliers) has no limit of its own: up to N = 170
 * (Cholesky) / 169 (LDL^T) a program's KKT matrix is factored in shared memory, above that by blocked
 * kernels, as long as the batch's 2 N^2 doubles per program (with multipliers, 1 N^2 without) fit in
 * device memory. LMI cones keep their own limits (order <= 64), which BatchMaximize refuses (-1). */
void* CONEXB200_CreateBatch(void* const* programs, int count);
void CONEXB200_DeleteBatch(void* batch);
int CONEXB200_BatchMaximize(void* batch, const double* b, const CONEX_SolverConfiguration* config, double* y,
                            int* solved);
/* Per-program iteration counts and final by / cx / inv_sqrt_mu (any pointer may be NULL). */
void CONEXB200_BatchGetResults(void* batch, int* iterations, double* by, double* cx, double* inv_sqrt_mu);
/* Device time of the last batched solve and of its Newton steps (CUDA events). */
double CONEXB200_BatchMilliseconds(void* batch);
int CONEXB200_BatchStepMilliseconds(void* batch, double* out, int capacity);
/* Scaled dual variable of constraint `cone` of program `program` (like CONEX_GetDualVariable, same
 * numbering); returns its size. Equality blocks have none: nothing is written, the return value is 0. */
int CONEXB200_BatchGetDualVariable(void* batch, int program, int cone, double* x);
/* Replaces columns [first, first + count) of the data of constraint `constraint` (numbered like
 * CONEX_GetDualVariable, equality blocks included) in every program of the batch. Cones on all m variables:
 * column j < m holds the coefficients of y_j (LP: column j of A; SOC: column j of the (n + 1) x m A; LMI:
 * vec(A_j)), column m the affine term (c / C). Cones on a list of m_k variables v: column j < m_k holds the
 * coefficients of y[v_j], column m_k the affine term. Equality blocks: column j < nvars is column j of A,
 * column nvars is b.
 * data: host memory, B blocks of rows x count column-major (program p at data + p * rows * count).
 * Returns 0, or -1 on bad arguments (the batch is then unchanged). The next BatchMaximize uses the new data;
 * a warm start continues from the iterate of the previous solve. */
int CONEXB200_BatchUpdateConstraintData(void* batch, int constraint, int first, int count, const double* data);
/* The shape of that data for constraint `constraint`: *rows (cones: n for LP, n + 1 for SOC, n * n for LMI; equality
 * blocks: their rows) and *columns (cones: m_k + 1 for a cone on m_k variables, m + 1 on all of them; equality
 * blocks: nvars + 1). Returns 0, or -1 when the batch has no
 * such constraint. The caller of CONEXB200_BatchUpdateConstraintData must pass blocks of exactly these rows. */
int CONEXB200_BatchConstraintDataShape(void* batch, int constraint, int* rows, int* columns);

#ifdef __cplusplus
}
#endif
#endif

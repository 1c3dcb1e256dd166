/*
 * cosmo_b200.h -- C ABI of the B200-native ADMM iteration engine that drops in
 * behind COSMO.jl's `COSMO.optimize!` hot loop.
 *
 * Boundary (reference file:line, COSMO.jl v0.8.11):
 *   - the engine owns everything between `allocate_loop_variables!` / the
 *     operator warm start (src/solver.jl:125-129) and `recover_mu!` at loop
 *     exit (src/solver.jl:167); `setup!` (src/setup.jl:18-64: Ruiz scaling,
 *     row ranges) stays upstream and `reverse_scaling!` /
 *     `reverse_decomposition!` (src/solver.jl:179-190) stay downstream, in
 *     unchanged host code.
 *   - per-plugin entry points mirror the reference's own seams:
 *       AbstractKKTSolver  ctor / solve! / update_rho! / free_memory!
 *                          (src/linear_solver/kktsolver.jl:5-13, 310-313)
 *       AbstractConvexSet  project!(x, set)          (src/convexset.jl:885-891)
 *
 * Conventions
 *   - plain pointers and sizes only; every array argument is a HOST pointer
 *     owned by the caller (Julia GC memory under GC.@preserve). The engine
 *     copies inputs to HBM inside the call and never keeps a host pointer.
 *   - matrices arrive exactly as Julia stores them: SparseMatrixCSC{T,Int64},
 *     1-based colptr/rowval (`index_base = 1`); `index_base = 0` accepts
 *     SciPy-style 0-based int64 arrays.
 *   - `dtype` selects Float64 / Float32 models (Model{Float64}, Model{Float32}).
 *   - every function returns 0 on success or a negative COSMO_B200_ERR_* code;
 *     `cosmo_b200_last_error` returns the message (the Julia shim rethrows it as
 *     ErrorException). Solver outcomes are NOT errors: they are reported in
 *     `cosmo_b200_result.status` (1:1 with the reference's status Symbols,
 *     src/solver.jl:113,161,175,311-353).
 *   - one host thread per handle; `solve` is synchronous.
 */
#ifndef COSMO_B200_H
#define COSMO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define COSMO_B200_ABI_VERSION 4

typedef struct cosmo_b200_handle cosmo_b200_handle;

/* cosmo_b200_problem.flags */
#define COSMO_B200_PROBLEM_EQUILIBRATE 1 /* run scale_ruiz! on the device (data handed over unscaled) */

enum {
  COSMO_B200_OK = 0,
  COSMO_B200_ERR_INVALID = -1,     /* bad argument / dimension mismatch (interface.jl:369-392) */
  COSMO_B200_ERR_UNSUPPORTED = -2, /* unknown set type, BigFloat, unsupported option: shim falls back to Julia */
  COSMO_B200_ERR_CUDA = -3,        /* CUDA runtime error or no usable sm_100 device */
  COSMO_B200_ERR_ALLOC = -4,
  COSMO_B200_ERR_NCCL = -5,
  COSMO_B200_ERR_NUMERICAL = -6    /* eigensolver failed to converge (LAPACK info != 0, convexset.jl:186) */
};

enum { COSMO_B200_F64 = 0, COSMO_B200_F32 = 1 };

/* cone types in `sort_sets` order (src/interface.jl:466-475) */
enum {
  COSMO_B200_ZERO = 0,         /* ZeroSet,          convexset.jl:16-28   */
  COSMO_B200_NONNEG = 1,       /* Nonnegatives,     convexset.jl:52-74   */
  COSMO_B200_BOX = 2,          /* Box(l,u),         convexset.jl:803-847 */
  COSMO_B200_SOC = 3,          /* SecondOrderCone,  convexset.jl:92-114  */
  COSMO_B200_PSD_SQUARE = 4,   /* PsdCone / DensePsdCone,                 convexset.jl:271-321 */
  COSMO_B200_PSD_TRIANGLE = 5, /* PsdConeTriangle / DensePsdConeTriangle, convexset.jl:362-412 */
  /* 3-d cones (sort_sets puts every remaining type in class 6 too, interface.jl:473) */
  COSMO_B200_EXP = 6,          /* ExponentialCone,      convexset.jl:497-618 */
  COSMO_B200_DUAL_EXP = 7,     /* DualExponentialCone,  convexset.jl:749-789 */
  COSMO_B200_POW = 8,          /* PowerCone(alpha),     convexset.jl:625-742 */
  COSMO_B200_DUAL_POW = 9,     /* DualPowerCone(alpha), convexset.jl:765-789 */
  COSMO_B200_PSD_TRIANGLE_COMPLEX = 10 /* PsdConeTriangle{T, Complex{T}}(dim), dim = N^2 (convexset.jl:344-360,444-490);
                                          projected through the real 2N x 2N embedding [[A, -B], [B, A]]: in shared
                                          memory up to N = 48, through the large-cone path (tensor cores) beyond */
};

/* status (src/solver.jl:113,161,175,311-353) */
enum {
  COSMO_B200_UNDETERMINED = 0,
  COSMO_B200_SOLVED = 1,
  COSMO_B200_MAX_ITER_REACHED = 2,
  COSMO_B200_TIME_LIMIT_REACHED = 3,
  COSMO_B200_PRIMAL_INFEASIBLE = 4,
  COSMO_B200_DUAL_INFEASIBLE = 5,
  COSMO_B200_UNSOLVED = 6
};

/* accelerators (COSMOAccelerators.jl types selectable through settings.accelerator) */
enum { COSMO_B200_ACC_EMPTY = 0, COSMO_B200_ACC_ANDERSON = 1 };

/* KKT plugins (src/linear_solver/kktsolver_indirect.jl:173-189; kktsolver.jl:285-349) */
enum {
  COSMO_B200_KKT_CG = 0,             /* CGIndirectKKTSolver      (reduced system, CG)      :3-88   */
  COSMO_B200_KKT_MINRES_REDUCED = 1, /* IndirectReducedKKTSolver(solver_type = :MINRES)    :3-88   */
  COSMO_B200_KKT_MINRES = 2,         /* MINRESIndirectKKTSolver  (full KKT, MINRES)        :90-162 */
  COSMO_B200_KKT_DIRECT = 3          /* the engine's counterpart of QdldlKKTSolver / CholmodKKTSolver (kktsolver.jl:285-349):
                                        exact solves through a dense fp64 Cholesky factor of the reduced matrix
                                        P + sigma I + A' diag(rho) A, factored at create and again after every change of
                                        rho or sigma.  Chosen at create; single-GPU; refused (ERR_UNSUPPORTED) when the
                                        factor would need more than half of the free device memory, and with
                                        "Objective function is not convex." (ERR_INVALID) when the matrix is not
                                        positive definite. */
};

/* SparseMatrixCSC{T,Int64} as Julia stores it */
typedef struct {
  int64_t nrows, ncols;
  const int64_t* colptr; /* ncols+1 */
  const int64_t* rowval; /* nnz */
  const void* nzval;     /* nnz, dtype */
} cosmo_b200_csc;

/* one entry of CompositeConvexSet.sets (src/projections.jl:20-31) */
typedef struct {
  int32_t type;     /* COSMO_B200_ZERO ... */
  int32_t max_iter; /* Exp/Pow cones: MAX_ITER of the projection (0 = reference default, 100 / 20) */
  int64_t dim;      /* rows of this set (for PSD: length of the vector, N^2 or N(N+1)/2; Exp/Pow: 3) */
  const void* l;    /* Box only: lower/upper bounds, already scaled by E (convexset.jl:863-867) */
  const void* u;
  double alpha;     /* PowerCone / DualPowerCone exponent in (0,1), convexset.jl:631-634 */
  double tol;       /* Exp/Pow cones: EXP_TOL / POW_TOL (0 = reference default 1e-8) */
} cosmo_b200_set;

/* ws.p (ProblemData, types.jl:158-175) + ws.sm (ScaleMatrices, types.jl:130-151) after setup! */
typedef struct {
  int32_t dtype;      /* COSMO_B200_F64 | COSMO_B200_F32 */
  int32_t index_base; /* 1 = Julia, 0 = C */
  int32_t device;     /* CUDA device ordinal */
  int32_t flags;      /* COSMO_B200_PROBLEM_* */
  int64_t m, n;
  cosmo_b200_csc P; /* n x n, both triangles stored */
  cosmo_b200_csc A; /* m x n, model form A x + s = b */
  const void* q;    /* n */
  const void* b;    /* m */
  int64_t n_sets;
  const cosmo_b200_set* sets;
  /* diagonal scalings (NULL => identity).  With flags & COSMO_B200_PROBLEM_EQUILIBRATE and settings.scaling != 0 they
     must be NULL: (P, q, A, b) and the Box bounds are UNSCALED and the engine equilibrates them on the device
     (scale_ruiz!, scaling.jl:21-116); the host then reads D, E, c back with cosmo_b200_get_scaling for
     scale_variables! / reverse_scaling!. */
  const void* D;
  const void* Dinv;
  const void* E;
  const void* Einv;
  double c; /* cost scaling ws.sm.c[] (1.0 when unscaled) */
} cosmo_b200_problem;

/* COSMO.Settings (src/settings.jl:61-155), the fields the loop reads */
typedef struct {
  double rho, sigma, alpha;
  double eps_abs, eps_rel, eps_prim_inf, eps_dual_inf;
  int64_t max_iter;
  int32_t check_termination, check_infeasibility;
  int32_t scaling; /* != 0: residuals are unscaled with Einv / cinv*Dinv (residuals.jl:43-49) */
  int32_t adaptive_rho;
  int32_t adaptive_rho_interval; /* 0 = automatic: chosen once (time in the loop) > adaptive_rho_fraction * setup_time,
                                    rounded to a multiple of check_termination (solver.jl:244-256) */
  int32_t kkt_solver;            /* COSMO_B200_KKT_* */
  double adaptive_rho_tolerance;
  int64_t adaptive_rho_max_adaptions;
  double RHO_MIN, RHO_MAX, RHO_TOL, RHO_EQ_OVER_RHO_INEQ, COSMO_INFTY, MIN_SCALING;
  double time_limit;
  double tol_constant, tol_exponent; /* kktsolver_indirect.jl:21,168-170 */
  int32_t verbose;                   /* bit 0: settings.verbose (iteration log), bit 1: settings.verbose_timing */
  int32_t psd_max_sweeps;            /* Jacobi eigensolver sweep cap (engine-specific) */
  /* accelerator (settings.jl:96-98,136-138; accelerator_interface.jl:58-114) */
  int32_t accelerator;         /* COSMO_B200_ACC_EMPTY | COSMO_B200_ACC_ANDERSON (Type2{QRDecomp}, RestartedMemory,
                                  NoRegularizer, ImmediateActivation) */
  int32_t accelerator_mem;     /* history length `mem` (reference default 15) */
  int32_t accelerator_min_mem; /* columns needed before a candidate is formed (package default 3) */
  int32_t safeguard;           /* settings.safeguard */
  double safeguard_tol;        /* settings.safeguard_tol (2.0) */
  /* ABI 3 */
  double adaptive_rho_fraction; /* settings.adaptive_rho_fraction (0.4), used by the automatic interval rule */
  double setup_time;            /* seconds the host spent in setup! (ws.times.setup_time: scaling, decomposition, the creation
                                   of this engine); 0: the engine uses its own creation time.  Feeds the automatic rho
                                   interval and the time limit, which the reference measures from before setup!
                                   (solver.jl:119,349) */
  double MAX_SCALING;           /* settings.MAX_SCALING (1e4), read by the device equilibration */
  /* ABI 4 */
  double obj_true;              /* settings.obj_true (NaN = off): has_converged additionally requires
                                   |obj_true - cost| <= obj_true_tol at a termination check (residuals.jl:127-140) */
  double obj_true_tol;          /* settings.obj_true_tol (1e-3) */
} cosmo_b200_settings;

/* COSMO.Result / ResultInfo / ResultTimes (types.jl:26-41, 65-71, 93-112) */
typedef struct {
  /* caller-allocated outputs in the SCALED coordinates the loop works in
     (ws.vars.x = view(w_prev,1:n), ws.vars.s.data, ws.vars.mu at solver.jl:167);
     reverse_scaling! stays in host code. Any of them may be NULL. */
  void* x;  /* n */
  void* s;  /* m */
  void* mu; /* m  (y = -mu) */
  double obj_val;
  int64_t iter;
  int64_t safeguarding_iter;
  int32_t status;
  int32_t _pad;
  double r_prim, r_dual, max_norm_prim, max_norm_dual;
  double rho; /* final scalar rho (ws.rho) */
  double* rho_updates;      /* optional caller buffer for ws.rho_updates */
  int64_t rho_updates_cap;
  int64_t n_rho_updates;
  /* times in seconds (ResultTimes, types.jl:26-41).  proj_time = device time of admm_z! (solver.jl:15,152; here fused
     with the right-hand side of admm_x!), kkt_time = device time of the KKT solves incl. the fused ADMM tail: CUDA
     events on the engine stream, filled when settings.verbose bit 1 is set or the problem is not latency-bound
     (n + m >= 20000 or a large PSD cone), 0 otherwise; res_time = host time inside the termination checks. */
  double solver_time, setup_time, iter_time, proj_time, kkt_time, res_time;
  double iter_time_device; /* the loop timed with CUDA events on the engine stream */
  /* statistics */
  int64_t kkt_inner_iterations; /* CG / MINRES iterations summed over the solve */
  int64_t kkt_multiplications;  /* reduced / full operator applications (S.multiplications) */
  int64_t kernel_launches;      /* engine kernels launched inside the loop */
} cosmo_b200_result;

/* ---- lifecycle ---------------------------------------------------------- */
int cosmo_b200_abi_version(void);
/* COSMO.Settings{T}() defaults (settings.jl:101-139) with kkt_solver = CG and accelerator = COSMO_B200_ACC_EMPTY
   (the reference default is the Anderson accelerator, settings.jl:136-138: set accelerator = COSMO_B200_ACC_ANDERSON;
   the Julia shim of INTEGRATION.md copies it from ws.accelerator) */
int cosmo_b200_default_settings(cosmo_b200_settings* out);
/* _make_kkt_solver! + Variables{T}(m,n,C) + classify_constraints! + set_rho_vec!
   (setup.jl:1-7,75-85; types.jl:263-279; parameters.jl:3-13): uploads the problem. */
int cosmo_b200_create(cosmo_b200_handle** out, const cosmo_b200_problem* prob, const cosmo_b200_settings* settings);
/* free_memory!(ws) (solver.jl:205-208) */
void cosmo_b200_destroy(cosmo_b200_handle* h);
/* last error message of a handle (or of the failed create when h == NULL) */
const char* cosmo_b200_last_error(const cosmo_b200_handle* h);

/* ---- model updates ------------------------------------------------------ */
int cosmo_b200_update_settings(cosmo_b200_handle* h, const cosmo_b200_settings* settings);
/* warm_start_primal!/slack!/dual! (interface.jl:117-179), already scaled; NULL = leave unchanged */
int cosmo_b200_warm_start(cosmo_b200_handle* h, const void* x, const void* s, const void* mu);
/* update!(model, q=, b=) (interface.jl:187-211), already scaled; NULL = leave unchanged */
int cosmo_b200_update_qb(cosmo_b200_handle* h, const void* q, const void* b);
/* update_rho!(kkt_solver, rho_vec) (kktsolver_indirect.jl:164-166): overrides the row penalties */
int cosmo_b200_update_rho(cosmo_b200_handle* h, const void* rho_vec, double rho);
/* empty_model!-like reset of iterates, rho, CG warm start and call counter */
int cosmo_b200_reset(cosmo_b200_handle* h);

/* ---- the hot loop (solver.jl:125-167) ------------------------------------ */
int cosmo_b200_solve(cosmo_b200_handle* h, cosmo_b200_result* out);

/* ---- plugin-granularity entry points (also the parity-test hooks) -------- */
/* project!(s, C): s_out = Pi_K(w_s) (convexset.jl:885-891) */
int cosmo_b200_project(cosmo_b200_handle* h, const void* w_s, void* s_out);
/* solve!(kkt_solver, sol, rhs): rhs, sol in R^{n+m} (kktsolver_indirect.jl:36-88,123-162; kktsolver.jl:315-320);
   inner_iterations = 0 for the direct solver */
int cosmo_b200_kkt_solve(cosmo_b200_handle* h, const void* rhs, void* sol, int64_t* inner_iterations);
/* calculate_residuals! + max_res_component_norm + calculate_cost! (residuals.jl:30-96,143-147)
   for given (x, s, mu); out = {r_prim, r_dual, max_norm_prim, max_norm_dual, cost} */
int cosmo_b200_residuals(cosmo_b200_handle* h, const void* x, const void* s, const void* mu,
                         int32_t ignore_scaling, double out[5]);
/* y = M x for M in {0: A, 1: A', 2: P} (the mul! calls at kktsolver_indirect.jl:53-63) */
int cosmo_b200_spmv(cosmo_b200_handle* h, int32_t which, const void* x, void* y);
/* time `reps` back-to-back launches of one SpMV kernel with CUDA events; returns ms per launch */
int cosmo_b200_spmv_bench(cosmo_b200_handle* h, int32_t which, int32_t reps, double* ms_per_launch,
                          double* algorithmic_bytes);
/* read back the current per-row penalty vector (ws.rho_vec) */
int cosmo_b200_get_rho_vec(cosmo_b200_handle* h, void* rho_vec);
/* ws.sm.D.diag (n), ws.sm.E.diag (m), ws.sm.c[] as used by the engine: what the host passed at create, or what the
   device equilibration computed (scaling.jl:21-116); all ones when settings.scaling == 0.  NULL pointers are skipped. */
int cosmo_b200_get_scaling(cosmo_b200_handle* h, void* D, void* E, double* c);
/* read back the operator variable w = [w_x; w_s] (n+m) */
int cosmo_b200_get_w(cosmo_b200_handle* h, void* w);

/* ---- multi-GPU (one process per GPU; rows sharded, n-vectors replicated) -- */
/* 128-byte ncclUniqueId created on rank 0 and broadcast by the host plumbing */
int cosmo_b200_comm_unique_id(void* id128);
int cosmo_b200_comm_init(cosmo_b200_handle* h, int32_t nranks, int32_t rank, const void* id128);
/* Peer-memory exchange over NVLink/NVSwitch for the reduced-KKT operator partials (optional; replaces
   the per-application NCCL allreduce by a one-shot sum fused into the consumer kernels).
   export: 128 bytes (two CUDA IPC handles) per rank; the host all-gathers them in rank order;
   attach: maps the peers' buffers.  All ranks must be on one NVLink-connected node. */
int cosmo_b200_comm_p2p_export(cosmo_b200_handle* h, void* blob128);
int cosmo_b200_comm_p2p_attach(cosmo_b200_handle* h, const void* blobs, int32_t nranks);

/* ---- diagnostics ---------------------------------------------------------- */
/* Which path projected the large PSD cones (N > 96) so far: out = {tensor-core projections, tensor-core fallbacks to
   block Jacobi, Newton-Schulz steps of the last one, weighted-residual checks of the last one, FP64-FMA sign
   projections, their fallbacks, block-Jacobi sweeps of the last eigensolve, int8 slices per operand}. */
int cosmo_b200_psd_stats(cosmo_b200_handle* h, int64_t out[8]);
/* The direct KKT solver's factorisations (ws.times.init_factor_time / factor_update_time, types.jl:31-32):
   factorizations = number of factorisations so far; seconds[0] = device time of the initial one (at create),
   seconds[1] = device time of all later ones (after rho / sigma changes), assembly of the reduced matrix included.
   A handle on an indirect solver reports 0 and zeros. */
int cosmo_b200_kkt_factor_stats(cosmo_b200_handle* h, int64_t* factorizations, double seconds[2]);
/* Symbolic analysis of the full quasi-definite KKT matrix K = [P + sigma I, A'; A, -R^-1] (the pattern QdldlKKTSolver
   factors, kktsolver.jl:285-320): approximate minimum degree ordering with dense nodes ordered last, elimination tree,
   column counts, relaxed supernodes.  Host only: needs no GPU and no handle, reads only the problem's dimensions,
   index_base and the patterns of P and A (no duplicate entries).  perm (n + m entries, or NULL) receives the
   elimination order, 0-based: perm[k] is the k-th node eliminated (node j < n is x_j, node n + i is row i of A).
   info = {nnz(L) including the diagonal, supernodes, height of the supernodal tree, widest supernode (columns),
   largest front (columns + rows below), factor bytes (fp64 (columns + rows below) x columns per supernode),
   workspace bytes (fan-in panel, solve vectors, scatter map), nodes postponed as dense}.  The byte counts are those of
   a supernodal factorisation on the device (DESIGN §3d), which the engine does not have yet.
   Errors through cosmo_b200_last_error(NULL). */
int cosmo_b200_kkt_symbolic(const cosmo_b200_problem* prob, int64_t* perm, int64_t info[8]);
/* The product kernel of the large-cone PSD projection on its own: C = A B for symmetric, commuting N x N fp64
   matrices (column-major) through `k` int8 slices on tcgen05 (csrc/tc_gemm.cuh; the reference's counterpart is the
   BLAS-3 part of project!(::PsdCone), convexset.jl:244-260).  `groups` = number of slice-pair groups kept
   (0: the default of `k`); supported (k, groups): (8,10) (8,8) (7,7) (6,8) (4,6); `reserved` must be 0.
   frob2 = {|C|_F^2, |I - C|_F^2} from the fused reductions.
   No handle: uses the current device.  Errors through cosmo_b200_last_error(NULL). */
int cosmo_b200_tc_gemm_test(int32_t N, int32_t k, int32_t groups, int32_t reserved, const double* A, const double* B, double* C,
                            int32_t reps, double* ms_per_product, double* frob2);

#ifdef __cplusplus
}
#endif
#endif /* COSMO_B200_H */

/* mgbx.h -- C ABI of libmgbx.so: the B200-native (sm_100a) barrier-Newton engine.
 *
 * This is the drop-in boundary for the hot path of sloisel/MultiGridBarrier.jl.  The reference
 * selects a backend with a `Device` marker and moves a pure-data `MGBProblem` across with
 * `native_to_device(device, prob)` (src/device.jl:18-60, src/mgb.jl:798-842); the solve then runs
 * `mgb_driver -> mgb_core -> mgb_step -> newton -> barrier f0/f1/f2` on backend arrays.  A Julia
 * `B200Device` shim (INTEGRATION.md) or the Python host mirror (multigridbarrier.jl_b200/) binds
 * exactly the entry points below by `ccall` / `ctypes`:
 *
 *   mgbx_create        <- native_to_device(::Type{CUDADevice}, prob)   ext/MultiGridBarrierCUDAExt/conversion.jl:152-159
 *   mgbx_step          <- mgb_step (+ newton, line search, f0/f1/f2, R'HR, solve)   src/mgb.jl:16-82, src/newton.jl:227-287
 *   mgbx_scalars       <- the scalars mgb_core / mgb_driver read between t-steps   src/mgb.jl:135-136,454,526-527
 *   mgbx_phase1_init   <- feasibility probe + slack initialisation    src/mgb.jl:417-448
 *   mgbx_attach_feasibility <- M[2] of native_to_device, moved only if phase I runs   src/mgb.jl:449-452
 *   mgbx_set_feasibility_box <- _feasibility_convex(Q, b, R, ...)     src/mgb.jl:217-287,504
 *   mgbx_handoff       <- z2 = SOL_feas.z[1:len]                      src/mgb.jl:566
 *   mgbx_matched_t     <- _matched_t                                  src/mgb.jl:307-330
 *   mgbx_get_z / mgbx_set_z <- device_to_native / warm starts         src/mgb.jl:841
 *   mgbx_get_z_unfinalized  <- SOL.z_unfinalized                      src/mgb.jl:76-80
 *   mgbx_destroy       <- mgb_cleanup                                 src/mgb.jl:840
 *   mgbx_barrier_eval, mgbx_hessian_pattern, mgbx_hessian_values, mgbx_solve_newton_system,
 *   mgbx_plan_pattern, mgbx_recover_transfer, mgbx_kron_factor, mgbx_shard_row_range  <- fine-grained parity hooks for barrier(Q).f0/f1/f2 (src/convex.jl:155-202),
 *                         _make_block_assembly_plan (src/BlockMatrices.jl:322-491) and solve (src/utils.jl:142-145)
 *
 * Conventions
 *   - plain pointers and sizes only; every array argument is HOST memory owned by the caller, the
 *     library copies what it needs at mgbx_create and owns all device memory behind the handle;
 *   - all matrices are column-major exactly as the Julia arrays are (an n x k grid is k contiguous
 *     columns of length n; BlockDiag.data is p x p x N, src/BlockMatrices.jl:17-27);
 *   - indices are 0-based int64 (Julia's Int minus one);
 *   - every call returns an int status: 0 ok, >0 numerical outcome (MGBX_NOT_CONVERGED ...),
 *     <0 error (argument / CUDA / allocation); no exceptions cross the ABI; the text of the last
 *     error is available from mgbx_last_error();
 *   - one handle <-> one CUDA stream <-> one host thread at a time (re-entrant across handles);
 *   - there is NO CPU fallback: without a CUDA device mgbx_create fails with MGBX_ERR_CUDA.
 */
#ifndef MGBX_H
#define MGBX_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MGBX_ABI_VERSION 2
#define MGBX_MAX_LEVELS 32
#define MGBX_MAX_ND 12      /* rows of D seen by one node functor (incl. phase-I extras) */
#define MGBX_MAX_PIECES 6
#define MGBX_MAX_NI 6       /* inputs of one piece */
#define MGBX_MAX_NC 8       /* rows of one piece (EP: nz) */

enum {
  MGBX_OK = 0,
  MGBX_NOT_CONVERGED = 1,   /* Newton / step did not converge (caller applies kappa -> sqrt(kappa)) */
  MGBX_NON_FINITE = 2,      /* the starting point of a Newton run is outside the barrier's domain */
  MGBX_ERR_ARG = -1,
  MGBX_ERR_CUDA = -2,
  MGBX_ERR_ALLOC = -3,
  MGBX_ERR_UNSUPPORTED = -4,
  MGBX_ERR_INTERNAL = -5
};

enum { MGBX_PIECE_EP = 0, MGBX_PIECE_LINEAR = 1 };
enum { MGBX_MAIN = 0, MGBX_FEAS = 1 };

/* sparse matrix, CSR, 0-based, column indices sorted within a row */
typedef struct {
  int64_t rows, cols;
  const int64_t *rowptr;   /* rows + 1 */
  const int64_t *colind;   /* nnz */
  const double *val;       /* nnz */
} mgbx_csr;

/* one convex piece: y -> A*y[idx] + b; EP: [q; s] in the power cone s >= |q|^p
 * (src/convex_euclidian_power.jl:446-452); LINEAR: every row > 0 (src/convex_linear.jl:216-222) */
typedef struct {
  int32_t kind;            /* MGBX_PIECE_EP | MGBX_PIECE_LINEAR */
  int32_t ni, nc;          /* inputs, rows (EP: nc == ni == nz) */
  const int32_t *idx;      /* ni D-row indices, 0-based; NULL = 0..ni-1 (Colon) */
  const double *A;         /* n x (nc*ni): row i holds vec(A_i) column-major */
  const double *b;         /* n x nc */
  const double *p;         /* n, EP only */
  const double *mu;        /* n, EP only */
} mgbx_piece;

/* Convex set = pieces + optional select grid (src/convex_piecewise.jl:158-160) */
typedef struct {
  int32_t npieces;
  const mgbx_piece *pieces;
  const double *select;    /* n x npieces or NULL (all pieces active everywhere) */
} mgbx_convex;

/* one AMG (src/multigrid.jl:278-288): geometry-level data + level->fine prolongations */
typedef struct {
  int64_t n, N;            /* broken nodes, elements; n = p*N */
  int32_t p, nu, nD, L;    /* nodes/element, state variables, rows of D, levels */
  const double *w;         /* n quadrature weights */
  int32_t nops;            /* distinct non-identity operators */
  const double *const *op_data;  /* nops arrays p x p x N (BlockDiag.data) */
  const int32_t *D_var;    /* nD: state variable of D row k */
  const int32_t *D_op;     /* nD: operator id, -1 = identity */
  const mgbx_csr *R_fine;  /* L entries, AMG.R_fine of the reference (src/multigrid.jl:278-288).  With T given only
                              R_fine[L-1] ((nu*n) x m_L) is read: the coarser ones are R_fine[l] = R_fine[l+1]*T[l] and
                              may be left zero-initialised.  With T == NULL all L entries are read */
  const mgbx_csr *T;       /* L-1 level transfers m_{l+1} x m_l with R_fine[l] = R_fine[l+1]*T[l], or NULL: the reference
                              discards them after composing R_fine (src/multigrid.jl:166-170), so the library recovers
                              them from R_fine[0..L-1] itself (selector rows / matching columns / normal equations,
                              csrc/host_sparse.hpp recover_transfer; mgbx_recover_transfer is the host-only hook) */
  const int64_t *var_offsets;    /* L x (nu+1): first column of variable k at level l, or NULL (needs all R_fine[l]):
                                    read off the block-diagonal structure of R_fine[l] */
  /* multi-GPU element partition (zero / NULL for a single-rank problem): this rank holds a contiguous block of
   * elements; n above is the LOCAL node count */
  int64_t n_global;              /* nodes of the whole mesh (the 1/n of the barrier average, src/convex.jl:155-164) */
  const int32_t *var_local;      /* nu flags: 1 = the variable's fine-level unknowns are node-local (`:full` space, R block
                                    == identity) and live only on the owning rank; 0 = shared (replicated, all-reduced) */
} mgbx_amg;

/* MGBProblem (src/mgb.jl:666-674) */
typedef struct {
  mgbx_amg amg[2];         /* [MGBX_MAIN], [MGBX_FEAS] (amg[1].n == 0: no phase-I data) */
  const double *f_grid;    /* n x nD(main) */
  const double *g_grid;    /* n x nu(main) */
  mgbx_convex Q;
  const double *barrier_weights; /* n (already normalised, 0 = node dropped) or NULL = 1/n */
} mgbx_problem;

typedef struct {
  int32_t dense_direct_max;  /* Newton systems with <= this many unknowns: dense Cholesky (default 2048) */
  int32_t coarse_max;        /* V-cycle is cut at the first level with <= this many unknowns (default 128 = the maximum) */
  int32_t pcg_maxit;         /* default 400 */
  double pcg_rtol;           /* relative residual, default 1e-7: Newton counts, the t-schedule and z are unchanged from 1e-9 down to 1e-6 on
                                the bench workload (profiles/r02a_rtol_sweep.jsonl), the oracle lab says the same (tools/inexact_newton_lab.py) */
  int32_t smoother_sweeps;   /* pre = post smoothing sweeps (Chebyshev degree), default 2 */
  int32_t condense;          /* 1 (default): eliminate node-local :full variables exactly before PCG */
  int32_t device;            /* CUDA device ordinal, -1 = current */
  int32_t verbose;
  int32_t profile;           /* 1: time every kernel launch with CUDA events on the handle's stream (mgbx_kernel_stats) */
  int32_t persistent;        /* must be 2: the only solve kernel, k_pcg2 (csrc/pcg2.cu); kept for callers that read it */
  int32_t tail_max;          /* V-cycle levels with <= this many unknowns run inside CTA 0 of the solve kernel (default 1200) */
  double pcg_rtol_final;     /* relative residual during the finalize pass (stopping_exact), default 1e-15 (i.e. to stagnation) */
  int32_t fused;             /* 1 (default): fused element kernels (operator blocks staged once in shared memory), with the
                                specialised kernel for the default (u, s) Euclidean-power family where it applies;
                                2: generic fused kernel only; 0: separate per-node and per-block kernels (always used
                                when a block does not fit in shared memory) */
  int32_t smoother;          /* V-cycle smoother of the solve kernel: 1 (default) Chebyshev of degree smoother_sweeps
                                with diagonal scaling on [lam/cheb_ratio, lam], lam = Gershgorin bound; 0 l1-Jacobi */
  double cheb_ratio;         /* default 8 (sweep in profiles/r01z_smoother_sweep.jsonl) */
  int32_t precond_fp32;      /* 1: the V-cycle (preconditioner) reads FP32 copies of the level matrices (8 instead of 12 bytes per
                                non-zero); the PCG operator, vectors and all reductions stay FP64.  0 off, 2 (default) automatic: only when
                                the level matrices together have >= 10 M non-zeros (they no longer fit the L2: V-cycle HBM-bound) */
  int32_t lambda_power;      /* -1 (default): automatic -- 6 when the top matrix averages more than 16 entries per row (3-D meshes), else 0;
                                > 0: that many power iterations on D^-1 A per level and Newton system (warm-started) replace the
                                Gershgorin bound of lambda_max in the Chebyshev interval (the bound stays as an upper clamp).  Measured on
                                hardware (fem3d 32^3, profiles/r02c_stagnation_3d.jsonl): 42 % fewer PCG iterations; none in 2-D */
  double pcg_fail_rtol;      /* a PCG solve that breaks down is a FAILED solve: the Newton run reports "not converged" (as a failed
                                factorisation would in the reference, src/utils.jl:142-145).  A solve that ends (stagnation / pcg_maxit)
                                with |r|/|b| above this AND with the direction's energy still growing (pcg_fail_etol) is INEXACT: its
                                direction is used (inexact Newton under the line search) but its decrement -- which a CG iterate
                                under-estimates -- may not end the Newton iteration; only the stagnation rule of stopping_exact may.
                                Both are counted in mgbx_step_result.solve_failures.  Default 1e-5: Newton counts are unchanged down
                                to 1e-7 and within +-1 at 1e-6 (tools/inexact_newton_lab.py) */
  double pcg_fail_etol;      /* for CG from x = 0, g.x_k = |x_k|_A^2 grows monotonically to the Newton decrement g.H^-1 g.  Late in
                                the t-ramp (conditioning ~ t^2) the residual norm can stall above pcg_fail_rtol although that
                                energy -- what the stop rule and the Armijo test consume -- has converged: a stagnated solve is
                                accepted when its last four iterations added less than this share of the energy.  Default 1e-8 */
  int32_t pcg_stall_window;  /* PCG stops when the residual has not improved by 0.1 % for this many iterations (default 100: late in a 3-D
                                ramp the residual plateaus for dozens of iterations before it drops -- with 25 the solves of fem3d 32^3 stopped
                                at |r|/|b| ~ 1e-3; the finalize pass uses 6) */
  int32_t direct_fallback;   /* 1 (default): a PCG solve that broke down or stayed inexact is redone by the dense Cholesky when the
                                system has <= 8192 unknowns */
  int32_t elem_bulk;         /* 1 (default): the fused element kernel stages each tile's operator slabs and node columns with
                                cp.async.bulk (one instruction per slab / block column, completion on an mbarrier) instead of one
                                8-byte cp.async per double; 0: the per-double path */
  int32_t shard_solve;       /* multi-GPU: 1 (default) the leading V-cycle levels with >= shard_min_rows unknowns are ROW-SHARDED over the
                                ranks inside the persistent solve kernel (peer stores over NVLink into CUDA-IPC-mapped exchange arenas,
                                cross-GPU flag barrier, csrc/pcg2.hpp); 0: every rank runs the whole solve (replicated) */
  int32_t shard_min_rows;    /* default 100000 */
  int32_t shard_min_nnz;     /* default 4000000: a level is sharded over N ranks only if nnz (1 - 1/N) >= this (a phase over it must
                                be long enough to pay for the cross-GPU barrier) */
  int32_t spectral_kron;     /* 1 (default): dense (spectral) discretisations whose operators and prolongations are Kronecker products
                                (spectral2d: :dx = kron(DX, I), R = kron(R1, R1), src/spectral2d.jl:22-35) assemble R'HR sum-factorised
                                (one small DMMA GEMM per block of variables instead of full n x n x n products); 0: unstructured GEMMs */
  int32_t uncondensed_pcg;   /* 0 (default): a fine-level Newton system that keeps a slack variable which can be eliminated neither
                                node-locally nor element-locally, or whose slack was eliminated element-locally (a slack in :broken_P1,
                                test/test_pure_p2.jl: exact, element by element, when cfg.condense = 1 on one GPU), and that has more
                                unknowns than the dense direct solver takes (8192, counted after the elimination) is refused with
                                MGBX_ERR_UNSUPPORTED; 1: run the V-cycle PCG on it anyway (slow to fail late in the t-ramp) */
  int32_t analytic_schur;    /* 1 (default): the node-local Schur complement of a slack that enters ONE Euclidean-power cone is formed in
                                closed form, (2/rho) I + (4/rho^2)(B/(A+B)) q q' with H_ss = A + B, instead of H_qq - H_qs H_sq / H_ss:
                                the subtraction cancels to O(1/t) relative and leaves no correct digit along q at t ~ 1e8 (the reduced
                                matrix turns indefinite, the PCG stalls).  0: numerical subtraction (the round-1 behaviour; the
                                specialised p-Laplace kernel always uses the closed form) */
} mgbx_config;

/* options of one mgb_step (src/mgb.jl:16-30; defaults src/mgb.jl:360-363) */
typedef struct {
  int32_t maxit;             /* 10000 */
  int32_t max_newton;        /* ceil(log2(-log2(eps)))+2 = 8 */
  int32_t initial_step;
  int32_t stop_kind;         /* 0 stopping_exact(theta), 1 stopping_inexact(lambda_tol, theta) */
  double stop_lambda_tol;
  double stop_theta;
  int32_t finalize;          /* 0 none, 1 stopping_exact(finalize_theta) */
  double finalize_theta;
  int32_t line_search;       /* 0 backtracking(beta, c1), 1 illinois(beta) */
  double ls_beta, ls_c1;
} mgbx_step_opts;

typedef struct {
  int32_t converged;
  int32_t its[MGBX_MAX_LEVELS];   /* Newton iterations per level (SOL.its) */
  double y;                       /* last objective value */
  double gnorm;                   /* last |g| */
  double inc;                     /* last Newton decrement squared */
  int32_t f01_evals, f2_evals, linear_solves, pcg_iters;
  double ms_f01, ms_f2, ms_solve; /* device time (CUDA events) spent per stage */
  int32_t solve_failures;         /* linear solves that broke down (Newton run abandoned) or stayed inexact (see pcg_fail_rtol) */
  int32_t its_finalize;           /* the part of its[L-1] spent in the finalize pass (the reference adds it into its[L], src/mgb.jl:76-80) */
  int32_t direct_fallbacks;       /* PCG solves redone by the dense direct solver (cfg.direct_fallback) */
} mgbx_step_result;

typedef struct {
  double c_dot_Dz;                     /* sum_j dot(w .* f[:,j], D_j z) */
  double var_max[MGBX_MAX_ND];         /* max over nodes of state variable k */
  double var_absmax[MGBX_MAX_ND];      /* max |.| */
  int32_t all_finite;
} mgbx_scalars_out;

typedef struct mgbx_handle mgbx_handle;

void mgbx_default_config(mgbx_config *cfg);
void mgbx_default_step_opts(mgbx_step_opts *o, int64_t n);
int mgbx_abi_version(void);
int mgbx_device_count(void);

int mgbx_create(const mgbx_problem *prob, const mgbx_config *cfg, mgbx_handle **out);
void mgbx_destroy(mgbx_handle *h);
const char *mgbx_last_error(const mgbx_handle *h);   /* h may be NULL: last create error */

/* Multi-GPU, one handle per rank/GPU (SURVEY.md section 8e): elements are partitioned across ranks (the host slices the
 * problem, multigridbarrier.jl_b200/partition.py); inside the library the partial sums over elements -- R'g, the assembled
 * Hessian values, objective / line-search / duality-gap scalars -- are combined with NCCL all-reduces on the handle's stream,
 * and every rank then runs the identical (deterministic) multigrid-PCG solve on the shared unknowns.  NCCL is loaded with
 * dlopen("libnccl.so.2") only when mgbx_comm_init is called.  Rank 0 obtains an id and the host broadcasts it. */
int mgbx_nccl_unique_id(char id[128]);
int mgbx_comm_init(mgbx_handle *h, int rank, int nranks, const char id[128]);   /* id == NULL: reuse the process-wide communicator
                                                                                  created by an earlier call with the same (rank, nranks) */
int mgbx_comm_finalize(void);

/* the hot path */
int mgbx_step(mgbx_handle *h, int which, double t, const mgbx_step_opts *o, mgbx_step_result *r);
int mgbx_scalars(mgbx_handle *h, int which, mgbx_scalars_out *out);

/* phase I (src/mgb.jl:417-566) */
int mgbx_phase1_init(mgbx_handle *h, int32_t *needs_phase1, double *b, double *zabsmax);
/* the feasibility AMG may be given at create time (amg[1]) or attached only when mgbx_phase1_init reports that
 * phase I is needed (saves its upload for feasible starts); after attaching, call mgbx_phase1_init again */
int mgbx_attach_feasibility(mgbx_handle *h, const mgbx_amg *feas);
int mgbx_set_feasibility_box(mgbx_handle *h, double b, double Rbox);
int mgbx_reset_feasibility_state(mgbx_handle *h);    /* z_feas <- (z_main, initial slack): no warm start between box rounds */
int mgbx_handoff(mgbx_handle *h);                    /* z_main <- leading block of z_feas */
int mgbx_matched_t(mgbx_handle *h, double t_default, double *t_out, double *tstar_out);

/* state I/O: z is the stacked state vector, length nu*n of the selected AMG */
int mgbx_get_z(mgbx_handle *h, int which, double *z_host);
int mgbx_set_z(mgbx_handle *h, int which, const double *z_host);
/* the state of the last successful mgbx_step BEFORE its finalize pass (SOL.z_unfinalized, src/mgb.jl:76-80) */
int mgbx_get_z_unfinalized(mgbx_handle *h, int which, double *z_host);
/* replace the cost / boundary-data grids in place (parabolic_solve re-assembly, src/Parabolic.jl:162-167) */
int mgbx_set_grids(mgbx_handle *h, const double *f_grid, const double *g_grid);

/* parity hooks.  level is 0-based; s has m_level entries.
 * order 0: out[0] = f0;  order 1: out[0..m) = f1;  values of f2 through mgbx_hessian_values. */
int64_t mgbx_level_size(mgbx_handle *h, int which, int level);
int mgbx_barrier_eval(mgbx_handle *h, int which, int level, double t, const double *s, int order,
                      double *out);
int mgbx_hessian_pattern(mgbx_handle *h, int which, int level, int64_t *nnz, int64_t *rowptr,
                         int64_t *colind);           /* rowptr/colind may be NULL to query nnz */
int mgbx_hessian_values(mgbx_handle *h, int which, int level, double t, const double *s, double *val);
int mgbx_solve_newton_system(mgbx_handle *h, int which, int level, double t, const double *s,
                             const double *rhs, double *x, int32_t *pcg_iters);

/* number of kernels launched through this handle so far (bench.py's gpu_launches) */
int64_t mgbx_launch_count(const mgbx_handle *h);

/* device memory held by the handle, by category (text, one line per category) and in total */
int mgbx_memory_report(mgbx_handle *h, char *buf, int64_t buflen, int64_t *total_bytes);

/* shape of the fine-level linear system and of the persistent solve kernel's plan (for roofline arithmetic);
 * zero-filled until the first fine-level Newton system has been solved */
typedef struct {
  int32_t condensed, nlev, nbig, bottom_dense, grid, threads;
  int64_t m[MGBX_MAX_LEVELS], nnz[MGBX_MAX_LEVELS], nnzT[MGBX_MAX_LEVELS];   /* active V-cycle levels, top first */
  int64_t assembly_terms;     /* padded terms of the element-block -> CSR gather */
  int64_t hblk_entries;       /* pairs * N * p * p */
  int64_t galerkin_terms;     /* padded terms of all Galerkin product gathers */
  double dgemm_flops;         /* FP64 tensor-core (DMMA) flops issued through this handle so far (spectral path) */
  int32_t nshard, nranks;     /* multi-GPU: leading V-cycle levels that are row-sharded over the ranks (0: replicated solve), ranks */
} mgbx_solver_info_t;
int mgbx_solver_info(mgbx_handle *h, int which, mgbx_solver_info_t *out);

/* per-kernel-class launch counts and (with profile on) summed device time in ms; names[k] are static strings.
 * Arrays must hold at least 32 entries. */
int mgbx_kernel_stats(mgbx_handle *h, int reset, int32_t *nclasses, const char **names, int64_t *launches, double *ms);
int mgbx_set_profile(mgbx_handle *h, int on);

/* host-only (no GPU needed): the reference assembly plan's output pattern for R'HR
 * (src/BlockMatrices.jl:344-446) from R (CSR, rows = nu blocks of N elements x p nodes). */
int mgbx_plan_pattern(const mgbx_csr *R, int64_t N, int32_t p, int32_t nu, int32_t nD,
                      const int32_t *D_var, int64_t *nnz, int64_t *rowptr, int64_t *colind);

/* host-only (no GPU needed): T with R_next * T = R_cur, exactly as mgbx_create recovers the level transfers when
 * mgbx_amg.T == NULL.  val / rowptr / colind may be NULL to query nnz (rowptr holds R_next->cols + 1 entries). */
int mgbx_recover_transfer(const mgbx_csr *R_next, const mgbx_csr *R_cur, int64_t *nnz, int64_t *rowptr, int64_t *colind,
                          double *val);

/* host-only (no GPU needed): classical Ruge-Stueben hierarchy of a sparse symmetric matrix K -- the prolongations P_0 (finest) ...
 * P_{levels-1} the reference obtains from the un-vendored AlgebraicMultigrid.jl, `ruge_stuben(K; max_coarse=2).levels[i].P`
 * (src/amg_prolongators.jl:16-18): classical strength (theta, default 0.25), first-pass RS C/F splitting, direct interpolation,
 * Galerkin P'KP, at most max_levels levels (10), coarsening stops at max_coarse unknowns.  csrc/host_amg.hpp; bitwise equal to the
 * Python host mirror's hierarchy.ruge_stuben (tests/test_abi_cpu.py).  mgbx_rs_get with NULL arrays queries the sizes. */
typedef struct mgbx_rs_hierarchy mgbx_rs_hierarchy;
int mgbx_rs_create(const mgbx_csr *K, int32_t max_coarse, int32_t max_levels, double theta, mgbx_rs_hierarchy **out);
int32_t mgbx_rs_levels(const mgbx_rs_hierarchy *H);
int mgbx_rs_get(const mgbx_rs_hierarchy *H, int32_t level, int64_t *rows, int64_t *cols, int64_t *nnz, int64_t *rowptr, int64_t *colind,
                double *val);
void mgbx_rs_destroy(mgbx_rs_hierarchy *H);

/* host-only (no GPU needed): is the dense (r1 r2) x (c1 c2) matrix M a Kronecker product kron(A, B) of an r1 x c1 and an r2 x c2 factor
 * (row-major outputs; the scale is fixed by taking B as the block through M's largest entry)?  This is the test mgbx_create applies to
 * the dense operators and prolongations of a spectral discretisation (:dx = kron(DX, I), R = kron(R1, R1), src/spectral2d.jl:22-35)
 * before it assembles R'HR sum-factorised (cfg.spectral_kron).  *is_kron = 0: A and B are left untouched. */
int mgbx_kron_factor(const double *M, int32_t r1, int32_t r2, int32_t c1, int32_t c2, int32_t col_major, double *A, double *B, int32_t *is_kron);

/* host-only (no GPU needed): rows [row_begin, row_end) of a V-cycle level that `rank` owns in the row-sharded multi-GPU solve
 * (cfg.shard_solve; csrc/pcg2.hpp pcg2_rank_rows -- the same arithmetic the persistent kernel's plan uses): the level's sliced-ELL
 * slices (32 / lanes_per_row rows each) are dealt in contiguous runs to the nranks * ctas_per_rank CTAs of all ranks.  The
 * reference has no multi-GPU code (src/mgb.jl:392-403 only points at an MPI package); the partition follows the north-star. */
int mgbx_shard_row_range(int64_t rows, int32_t lanes_per_row, int32_t ctas_per_rank, int32_t nranks, int32_t rank, int64_t *row_begin,
                         int64_t *row_end);

#ifdef __cplusplus
}
#endif
#endif /* MGBX_H */

/* amg_b200.h -- C ABI of the B200-native solve phase for async-multigrid's additive AMG cycles.
 *
 * The reference has no plugin/FFI API; its solve-phase boundary is a set of free C++ functions
 * called SPMD from inside one OpenMP parallel region (SURVEY.md 8b).  A GPU backend cannot sit at
 * the per-thread kernel signature, so the seam is one level up: per cycle and per solve, called
 * from a single host thread.  Every entry point below names the reference interface it replaces.
 *
 * Conventions: plain pointers and sizes only; all matrices are CSR with int32 indices and fp64
 * values, A_l diag-first (the reference's assumption, src/SMEM_Smooth.cpp:385-386); host pointers
 * unless a name ends in _dev; every function returns 0 on success and a negative AMGB_E* code
 * otherwise (never exit()s, unlike src/SMEM_Setup.cpp:1613-1615); amgb_last_error() gives text.
 * There is no CPU fallback: if no sm_100-class device / driver is present amgb_create fails.
 */
#ifndef AMG_B200_H
#define AMG_B200_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct amgb_ctx amgb_ctx;

enum {
   AMGB_OK = 0,
   AMGB_EINVAL = -1,   /* bad argument / call order */
   AMGB_ECUDA = -2,    /* CUDA runtime error (text in amgb_last_error) */
   AMGB_ENOMEM = -3,
   AMGB_ENCCL = -4,
   AMGB_ESTATE = -5    /* hierarchy incomplete / setup not called */
};

/* enumerators keep the reference's numeric values (src/Main.hpp:47-75) */
enum { AMGB_SMOOTH_JACOBI = 0, AMGB_SMOOTH_HYBRID_JGS = 2, AMGB_SMOOTH_SEMI_ASYNC_GS = 4, AMGB_SMOOTH_ASYNC_GS = 5,
       AMGB_SMOOTH_L1_JACOBI = 6,
       AMGB_SMOOTH_L1_HYBRID_JGS = 12 /* L1_HYBRID_JACOBI_GAUSS_SEIDEL: hybrid JGS divided by the l1 norms; BPX only -- the reference
                                         reaches it through the Parfor branch alone (src/SMEM_Solve.cpp:324-334, src/SMEM_Smooth.cpp:253-263) */ };
enum { AMGB_SOLVER_MULT = 0, AMGB_SOLVER_AFACX = 1, AMGB_SOLVER_MULTADD = 2, AMGB_SOLVER_BPX = 3,
       AMGB_SOLVER_ASYNC_AFACX = 5, AMGB_SOLVER_ASYNC_MULTADD = 6,
       AMGB_SOLVER_IEBPX = 16 /* IMPLICIT_EXTENDED_SYSTEM_BPX: amgb_solve_extended; hierarchy as for BPX */ };
enum { AMGB_CONVERGE_LOCAL = 0, AMGB_CONVERGE_GLOBAL = 1 };       /* src/Main.hpp LOCAL/GLOBAL */
enum { AMGB_MAT_A = 0, AMGB_MAT_P = 1, AMGB_MAT_R = 2 };

/* InputData fields the solve phase reads (src/Main.hpp:187-235; defaults src/SMEM_Main.cpp:64-104) */
typedef struct {
   int solver;                  /* AMGB_SOLVER_*                                   (-solver)            */
   int smoother;                /* AMGB_SMOOTH_*                                   (-smoother)          */
   double smooth_weight;        /* omega                                           (-smooth_weight)     */
   int num_pre_smooth_sweeps;   /* >0 with post>0 selects the symmetrised smoother (src/SMEM_Solve.cpp:305-317) */
   int num_post_smooth_sweeps;
   int num_fine_smooth_sweeps;
   int num_coarse_smooth_sweeps;
   int jgs_block_rows;          /* hybrid JGS: Gauss-Seidel inside contiguous blocks of this many rows, Jacobi
                                   across blocks (the reference's block is a thread's row range,
                                   src/SMEM_Smooth.cpp:567-581; SURVEY.md 5.9e) */
   int use_sell;                /* 1: sliced-ELL (C=32) storage for low-variance levels, 0: CSR only */
   int l2_persist;              /* 1: pin the coarse hierarchy in L2 with an access-policy window */
   int use_stream;              /* 1: warp-stream CSR kernel (each warp reduces chunks of <= 256 consecutive entries through
                                   shared memory) for every matrix not stored as sliced ELL whose rows average fewer than
                                   96 entries; 0, and those long-row matrices: vector-per-row CSR */
   int factor_level0;           /* 1 (synchronous Multadd with the symmetrised smoother only): P_0 / R_0 are uploaded PLAIN and the
                                   smoothing factors are applied on the fly, Pbar_0 e = (I - w D^-1 A_0)(P_0 e), Rbar_0 r = R_0 (r - w A_0 D^-1 r):
                                   the level-0 smoother and Rbar_0 then share ONE pass over A_0.  Same operator, rounding-level
                                   differences; the explicit products (src/SMEM_Setup.cpp:1173-1254) are what 0 uses */
   int coarse_solve;            /* 0: SMEM convention, the coarsest level contributes nothing to Multadd/AFACx (the reference's
                                   hypre_GaussElimSolve result is never used there, SURVEY.md 5.9c); 1: DMEM convention, direct solve
                                   on the coarsest level (src/DMEM_Add.cpp:262-264, src/DMEM_Mult.cpp:393; with AMGB_SOLVER_MULT: DMEM_MultCycle,
                                   src/DMEM_Mult.cpp:207, instead of SMEM's pre + post sweeps there) applied as a dense inverse; in the
                                   asynchronous solves (amgb_solve_async, amgb_dist_solve_async) the coarsest level's group then
                                   works like the others: restrict, solve directly (AddCycle), prolong, update */
   int sell_sigma;              /* > 1: SELL-C-sigma (rows sorted by length inside windows of sigma rows) for the
                                   non-stencil matrices whose padding then stays <= 25 %; 0/1: off */
   int stream_variant;          /* retired: must be 8, what amgb_default_options sets (the warp-stream kernel); any other value
                                   is refused by amgb_set_options with AMGB_EINVAL.  Kept so that the fields after it stay in place */
   int sell_uniform;            /* 1 (default): SELL-U, a lossless re-encoding of sliced-ELL slices whose entries take few distinct
                                   (column - row, value) pairs (constant-coefficient stencil levels): the kernel then streams the vectors
                                   only.  Same CSR semantics, a row's terms summed in another order; 0: off */
   /* options of the asynchronous solver (src/SMEM_Main.cpp:66,71,93; -async_type, -res_compute_type, -read_type) */
   int async_type;              /* 0 FULL_ASYNC (default): u += e with fp64 global reductions; 1 SEMI_ASYNC: a group's
                                   "u += e; u_k = u" is one critical section (omp lock, src/SMEM_Async_AMG.cpp:238-283) */
   int res_compute_type;        /* 0 LOCAL (default): every level group recomputes the whole fine residual from its own copy of u;
                                   1 GLOBAL (async Multadd only, src/SMEM_Main.cpp:650-660): the rows of level 0 are dealt to ALL CTAs,
                                   which smooth level 0 and recompute the shared residual on their slices (src/SMEM_Async_AMG.cpp:35-70,356-416) */
   int read_type;               /* 0 READ_SOL (default): groups share the solution u; 1 READ_RES: groups share the residual,
                                   r -= A_0 e (src/SMEM_Async_AMG.cpp:227-236,285-296), u assembled at the end (:416-426) */
   int lean_storage;            /* 1: a matrix stored as sliced ELL keeps no second (CSR) copy in HBM -- what lets the 512^3 hierarchy
                                   (2.7 G entries in the A_l alone) fit one 180 GB GPU.  (L1-)Jacobi smoothers only; the transposed
                                   product is then unavailable for those matrices.  0 (default): both copies */
   int factor_restriction;      /* 1 (with factor_level0; synchronous Multadd, symmetrised (L1-)Jacobi smoother, num_fine_smooth_sweeps = 1,
                                   one GPU): the restrictions R_l of the levels l >= 1 the cycle restricts from are uploaded PLAIN (P_l^T)
                                   too, and Rbar_l r = P_l^T (r - A_l diag(s) r) (s = w/d, or 1/l1) is applied on the fly: the pass over
                                   A_l that the level's smoother makes anyway writes t_l = r_l - A_l diag(s) r_l beside e_l = s o (r_l + t_l),
                                   then r_{l+1} = R_l t_l.  P_l stay the explicit Pbar_l.  Same operator, rounding-level differences;
                                   AMGB_EINVAL from amgb_setup where the algebra does not hold.  0 (default): explicit Rbar_l */
   int sell_window_epilogue;    /* 1 (default): the products with a SELL-C-sigma matrix (sell_sigma dividing 256) park every row sum in
                                   shared memory and apply the epilogue (operand loads, stores of y) in row order, coalesced, instead
                                   of at the row's sorted slot.  The same arithmetic per row: identical results; only the order of the
                                   fused per-CTA norm / dot partial sums differs.  0: the epilogue at the slot */
} amgb_options;

void amgb_default_options(amgb_options *opt);

/* ---- lifetime ------------------------------------------------------------------------------- */
int amgb_create(amgb_ctx **ctx, int device);
int amgb_destroy(amgb_ctx *ctx);
const char *amgb_last_error(const amgb_ctx *ctx);
/* number of kernels this context has launched so far (graph replays counted per node) */
long long amgb_launch_count(const amgb_ctx *ctx);

/* ---- hierarchy upload: replaces the pointers SMEM_Setup/InitAlgebra hand to the solve phase
 *      (all_data->matrix.A/P/R[l], src/SMEM_Setup.cpp:217-276).  Arrays are copied to HBM. ----- */
int amgb_set_num_levels(amgb_ctx *ctx, int num_levels);
int amgb_set_matrix(amgb_ctx *ctx, int kind /*AMGB_MAT_**/, int level, int nrows, int ncols, int nnz,
                    const int *row_ptr, const int *col_idx, const double *values);
int amgb_set_options(amgb_ctx *ctx, const amgb_options *opt);
/* allocates work vectors, scale arrays (A_diag = d/omega, L1 norms: src/SMEM_Setup.cpp:225-238),
 * optional SELL copies, CUDA graphs.  Must follow the uploads. */
int amgb_setup(amgb_ctx *ctx);

/* ---- vectors (all_data->vector.f[0] / u[0]) ----------------------------------------------- */
int amgb_set_rhs(amgb_ctx *ctx, const double *f_host);
int amgb_set_solution(amgb_ctx *ctx, const double *u_host /* NULL = zero */);
int amgb_get_solution(amgb_ctx *ctx, double *u_host);
int amgb_get_residual(amgb_ctx *ctx, double *r_host);

/* ---- per-op entry points (unit parity; ChebySetup/BPXCycle callers) --------------------- */
/* y = alpha*M*x + beta*b  -- SMEM_MatVec / SMEM_SpGEMV / SMEM_Residual / SMEM_Restrict
 * (src/SMEM_MatVec.cpp:123-259,302-378,394-408).  b may be NULL when beta == 0. */
int amgb_spgemv(amgb_ctx *ctx, int kind, int level, double alpha, const double *x, double beta,
                const double *b, double *y);
/* y = M^T x -- SMEM_MatVecT / SMEM_Restrict with -no_construct_R (src/SMEM_MatVec.cpp:325-408): restriction through
 * the interpolation matrix itself; x has M.nrows entries, y M.ncols. */
int amgb_spgemv_transpose(amgb_ctx *ctx, int kind, int level, const double *x, double *y);
/* SMEM_Smooth dispatcher (src/SMEM_Solve.cpp:264-377) on level `level`: u is in/out (ignored on
 * input when zero_guess != 0).  symmetric != 0 selects SMEM_Sync_Symmetric{,L1}Jacobi. */
int amgb_smooth(amgb_ctx *ctx, int level, int smoother, int symmetric, int sweeps, int zero_guess,
                const double *f, double *u);
/* Explicit Gauss-Seidel block list of the hybrid Jacobi / Gauss-Seidel smoother on one level: bounds[0] = 0 <= ... <=
 * bounds[nblocks] = rows of the level (empty blocks allowed: threads without rows).  Replaces the thread row ranges thread.A_ns / A_ne[level][tid] that PartitionGrids
 * (src/SMEM_Setup.cpp:954-959) hands to SMEM_Sync_HybridJacobiGaussSeidel (src/SMEM_Smooth.cpp:533-586): with the reference's own
 * ranges the device reproduces a run of the reference with that many threads per level.  nblocks = 0: back to the uniform
 * blocks of opt.jgs_block_rows.  Call after the level's matrix is uploaded; synchronous cycles and amgb_smooth only. */
int amgb_set_jgs_blocks(amgb_ctx *ctx, int level, int nblocks, const int *bounds);
/* sqrt(sum x_i^2) -- Parfor_Norm2 (src/Misc.cpp:296-309) */
int amgb_norm2(amgb_ctx *ctx, const double *x, int n, double *out);

/* ---- cycles ------------------------------------------------------------------------------- */
/* one application of the selected additive cycle to a residual, zero initial guess: c = B r.
 * SMEM_Sync_Add_Vcycle (Multadd/AFACx, src/SMEM_Sync_AMG.cpp:408-621, sequential meaning
 * src/SEQ_AMG.cpp:110-235) or SMEM_Sync_Parfor_BPXcycle (src/SMEM_Sync_AMG.cpp:147-294). */
int amgb_cycle(amgb_ctx *ctx, const double *r_host, double *c_host);

/* SMEM_Solve, synchronous branch (src/SMEM_Solve.cpp:93-252) on the resident f,u: cycles until
 * ||r||/||r0|| < tol or max_cycles.  relres_hist[0..*n_cycles] (caller provides max_cycles+1
 * doubles, may be NULL).  cheby_flag: Chebyshev acceleration of the cycle (:169-188) with mu,
 * delta from ChebySetup (src/SMEM_Cheby.cpp:48-49).  solve_seconds: device time of the loop. */
int amgb_solve_sync(amgb_ctx *ctx, double tol, int max_cycles, int cheby_flag, double mu, double delta,
                    double *relres_hist, int *n_cycles, double *solve_seconds);

/* EigsPower (src/SMEM_Cheby.cpp:410-518): extreme eigenvalues of B*A by `iters` steps of power iteration (second,
 * deflated pass for the minimum), B = the selected cycle from a zero guess.  ChebySetup then takes
 * mu = (max+min)/(max-min), delta = 2/(max+min) (src/SMEM_Cheby.cpp:48-49) -> amgb_solve_sync(cheby_flag = 1). */
int amgb_eigs_power(amgb_ctx *ctx, int iters, double *eig_min, double *eig_max);

/* Conjugate gradients preconditioned by the selected additive cycle from a zero guess (the reference reaches this through
 * hypre's PCG with its cycles as the preconditioner: -hypre_pcg, src/DMEM_Setup.cpp:129-167) on the resident f, u; the
 * solution is left in u.  r = f - A u, then per iteration z = B r, rho = (r, z), p = z + (rho / rho_old) p (p = z on the
 * first), q = A p, sigma = (p, q), u += (rho / sigma) p, r -= (rho / sigma) q, until ||r|| / ||r_0|| < tol or max_iters.
 * relres_hist[0..*iters] holds that recurrence residual (caller provides max_iters + 1 doubles, may be NULL); final_relres is
 * the true ||f - A u|| / ||r_0||, recomputed once (0 when r_0 = 0); solve_seconds the device time of the loop.
 * AMGB_EINVAL, before any launch, unless the preconditioner is a fixed symmetric operator: solver MULTADD or BPX, smoother
 * weighted or L1 Jacobi, Multadd with both or neither of pre / post smoothing (otherwise Rbar != Pbar^T); also for a
 * distributed context and max_iters < 0.  coarse_solve = 1 (DMEM's convention) is allowed.  A must be symmetric positive
 * definite -- the caller's contract, as for amgb_eigs_power: rho or sigma not positive and finite is a breakdown,
 * AMGB_ESTATE with the quantity and the iteration in amgb_last_error; *iters, the history and u then hold the completed
 * iterations.  Parity with hypre_PCGSolve itself is not pinned (hypre is not vendored). */
int amgb_solve_pcg(amgb_ctx *ctx, double tol, int max_iters, double *relres_hist, int *iters, double *final_relres,
                   double *solve_seconds);

/* SMEM_Async_Add_AMG (src/SMEM_Async_AMG.cpp:7-437) as ONE persistent cooperative kernel: each
 * level's correction chain owns a CTA group; groups share u through fp64 global atomics, no grid
 * barrier.  Stop rule: LOCAL = every group stops after num_cycles own corrections; GLOBAL = all
 * stop once every level has done >= num_cycles (CheckConverge, src/Misc.cpp:418-442).
 * corrections_per_level[num_levels] = local_num_correct; relres = final ||f-Au||/||r0||. */
int amgb_solve_async(amgb_ctx *ctx, int num_cycles, int converge_type, int *corrections_per_level,
                     double *relres, double *solve_seconds);

/* CTA groups of the persistent kernel, sized by the reference's work model (PartitionLevels / BALANCED_THREADS,
 * src/SMEM_Setup.cpp:770-868,1083-1160): cta_begin[num_levels + 1], *grid = total CTAs.  Valid after the first
 * amgb_solve_async. */
int amgb_async_groups(amgb_ctx *ctx, int *cta_begin, int *grid);

/* seconds every level group spent inside the last launch of the persistent kernel (its root's %globaltimer): the measured
 * side of the CTA-group balancing (the reference prints per-thread wall times the same way, src/SMEM_Main.cpp:800-870) */
int amgb_async_group_times(amgb_ctx *ctx, double *seconds /* num_levels */);
/* Host-only (no CUDA call; the CPU test suite interprets the result against the oracle): the PROGRAMS the persistent kernel
 * interprets for these options on a hierarchy of num_levels levels -- one list of operations per level group (restriction
 * chain, smoother, prolongation chain, "u += e; u_k = u", count / stop, residual; csrc/launch.h AsyncOpSym, 128 bytes each).
 * ops: caller's array of max_ops records; op_begin[num_levels + 1]. */
int amgb_async_program(const amgb_options *opt, int num_levels, int symmetric, int factor_level0, void *ops, int max_ops, int *op_begin);

/* SMEM_ExtendedSystemSolve with IMPLICIT_EXTENDED_SYSTEM_BPX, synchronous (`-solver iebpx`; src/SMEM_ExtendedSystem.cpp:9-836,
 * finish :777-817, ExtendedSystemImplicitMatVec :838-907) on the resident f: Chebyshev-accelerated (mu, delta from
 * ChebySetup) weighted / L1 Jacobi on the semi-definite extended ("generating") system over all levels, plain P and
 * R = P^T as for BPX.  Stops when the reference's iteration counter (which starts at 1; no iteration at all for
 * num_cycles <= 1) reaches num_cycles or, from the second iteration on, when the extended residual drops below
 * tol * r0_ext.  ext_hist[it], 1 <= it < *iters (caller provides max(num_cycles,2)+1 doubles, may be NULL) = relative
 * extended residual measured in iteration it; *iters = the reference's local_num_correct; ext_relres / relres = final
 * relative residuals of the extended system and of A x = f; the solution x = sum_l P^{0<-l} u_l is left in u
 * (amgb_get_solution). */
int amgb_solve_extended(amgb_ctx *ctx, double tol, int num_cycles, double mu, double delta, double *ext_hist, int *iters,
                        double *ext_relres, double *relres, double *solve_seconds);

/* The EXPLICIT form run ASYNCHRONOUSLY (`-solver async_eebpx`: EXPLICIT_EXTENDED_SYSTEM_BPX with async_flag = 1,
 * src/SMEM_ExtendedSystem.cpp:295-365 without its barriers, stop rule :636-652) on a ONE-level context whose A_0 is the assembled
 * extended matrix AA (smooth_weight = 1) and whose resident f is bb: one persistent cooperative kernel, a CTA = a thread's
 * contiguous nnz-balanced row range, chaotic Chebyshev-Jacobi relaxations with no barrier between CTAs.  The extended
 * iterate is left in u; iters_min / iters_max = fewest / most sweeps a CTA did; ext_relres recomputed after the launch. */
int amgb_solve_extended_async(amgb_ctx *ctx, double tol, int num_cycles, double mu, double delta, int *iters_min, int *iters_max,
                              double *ext_relres, double *solve_seconds);

/* The IMPLICIT form run ASYNCHRONOUSLY (`-solver async_iebpx`: SMEM_ExtendedSystemSolve with IMPLICIT_EXTENDED_SYSTEM_BPX and
 * async_flag = 1, src/SMEM_Main.cpp:309, async branches of src/SMEM_ExtendedSystem.cpp:305,365,474-479,636-652) on the resident
 * f, hierarchy as for amgb_solve_extended (solver BPX or IEBPX, weighted or L1 Jacobi, one GPU).  Set-up and finish are those
 * of amgb_solve_extended; in between, one launch of the persistent kernel in which every level k owns a CTA group (the
 * reference's thread group of level k) that rebuilds the z1 / z2 chains from the other groups' latest u_j (j >= k) and
 * e_j (j < k), forms r_k, takes its own Chebyshev step (its own omega recurrence from 2) and refreshes e_k, with no barrier
 * between groups.  Stop rule (:636-652): no iteration at all for num_cycles <= 1; a group publishes its sum r_k^2 from its
 * second iteration on; group 0 raises the converge flag once the sum of the published (possibly stale) contributions is below
 * tol * r0_ext; a group whose loc_iters reaches num_cycles counts itself done, and groups keep iterating until the flag is up
 * or every group is done.  iters[num_levels] = every group's final loc_iters; ext_relres / relres = final relative residuals
 * of the extended system and of A x = f; group_seconds[num_levels] (may be NULL) = time every group spent in the launch; the
 * solution x = sum_l P^{0<-l} u_l is left in u (amgb_get_solution).  AMGB_EINVAL, before any launch, on a distributed
 * context, for other smoothers or solvers, and when one cooperative wave holds fewer CTAs than levels. */
int amgb_solve_extended_implicit_async(amgb_ctx *ctx, double tol, int num_cycles, double mu, double delta, int *iters,
                                       double *ext_relres, double *relres, double *group_seconds, double *solve_seconds);
/* Host-only (no CUDA call): the per-group programs amgb_solve_extended_implicit_async hands the persistent kernel for these
 * options on num_levels levels (csrc/launch.h AsyncOpSym records; ops: caller's array of max_ops; op_begin[num_levels + 1]).
 * AMGB_EINVAL for smoothers other than weighted / L1 Jacobi and for more than 32 levels. */
int amgb_ext_async_program(const amgb_options *opt, int num_levels, void *ops, int max_ops, int *op_begin);

/* Drop-in for one whole SMEM_Solve call with HOST buffers (what SMEM_Main's run loop would call,
 * src/SMEM_Main.cpp:694-757): uploads f, zeroes u (InitSolve), runs the sync or async solve named
 * by opt.solver, downloads u. */
int amgb_smem_solve(amgb_ctx *ctx, const double *f_host, double *u_host, double tol, int num_cycles,
                    double *relres_hist, int *n_cycles, int *corrections_per_level, double *final_relres,
                    double *solve_seconds);

/* ---- setup step next to the path (SURVEY.md 8f-1).  EXPERIMENTAL: compiled, not yet validated on hardware. ----------------
 * SmoothTransfer (src/SMEM_Setup.cpp:1173-1254; its Eigen products :1256-1339) on the device: Pbar = G P and Rbar = P^T GT with
 * G = I - w D^-1 A (or the L1 form) from the diag-first A_l (n x n) and the plain P_l (n x nc), host CSR in, host CSR out in
 * the reference's product layout (descending columns, entry with column == row first, :1382-1423).  Either output may be
 * NULL.  The arrays of an amgb_host_csr are malloc'ed by the library: release them with amgb_host_csr_free.  `ctx` supplies
 * the device and stream; no hierarchy needs to be defined. */
typedef struct { int nrows, ncols, nnz; int *row_ptr; int *col_idx; double *values; } amgb_host_csr;
int amgb_smooth_transfer(amgb_ctx *ctx, int smooth_interp_type /* AMGB_SMOOTH_JACOBI | AMGB_SMOOTH_L1_JACOBI */, double smooth_weight,
                         int n, const int *A_row_ptr, const int *A_col_idx, const double *A_values,
                         int nc, const int *P_row_ptr, const int *P_col_idx, const double *P_values,
                         amgb_host_csr *Pbar, amgb_host_csr *Rbar);
void amgb_host_csr_free(amgb_host_csr *m);

/* ---- introspection used by bench.py ------------------------------------------------------- */
/* event-timed duration (ms) of `reps` back-to-back launches of the fine-level residual kernel
 * r = f - A_0 u (the dominant kernel), on the context's stream */
int amgb_time_residual(amgb_ctx *ctx, int reps, double *ms_per_launch);
int amgb_level_storage(amgb_ctx *ctx, int kind, int level, int *is_sell);
/* event-timed y = M x for one matrix of the hierarchy (tools/spmv_sweep.py).  use_scaled_values:
 * 0 the values, 1 the column-scaled values; A_l only: 2 the symmetrised smoother's pass e = s o (2x - (A diag(s)) x) of the
 * explicit cycle, 3 the factorised restriction's pass t = x - (A diag(s)) x, e = s o (x + t) (amgb_options.factor_restriction);
 * P_l only: 4 the prolongation's e_l += P_l e_{l+1} (in place) */
int amgb_time_spmv(amgb_ctx *ctx, int kind, int level, int use_scaled_values, int reps, double *ms_per_launch);
/* One product y = gamma c + rs o (beta b + beta2 b2 + alpha M x) + xself xs through the solve's SpMV kernels, host in / host out,
 * for tests of the kernel paths.  coef = {alpha, beta, gamma, beta2, xself}; b, c, rs, b2, xs may be NULL (term absent).
 * mode 0: y only; 1: also *sum = sum_i y_i^2; 2: also *sum = sum_i y_i w_i; 3 (use_scaled_values = 1, b given): also
 * y2 = w o (b + y).  *window_path (may be NULL): 1 when the window-staged SELL-C-sigma kernel ran (sell_window_epilogue) */
int amgb_spmv_probe(amgb_ctx *ctx, int kind, int level, int use_scaled_values, const double *coef, const double *x, const double *b,
                    const double *c, const double *rs, const double *b2, const double *xs, const double *w, int mode, double *y,
                    double *y2, double *sum, int *window_path);
/* slices stored in the SELL-U encoding (amgb_options.sell_uniform) and their (delta, mask, value) groups */
int amgb_sellu_stats(amgb_ctx *ctx, long long *slices, long long *groups);
/* Host-only probe of the SELL-U encoder (no CUDA call; CPU test suite): CSR + column-scaled values in; out, per slice, the
 * first group and the group count (2 ints per slice; count 0 = slice not encoded) into the DEDUPLICATED group table, and the
 * table's delta / lane mask / value / scaled value (malloc'ed: release with amgb_host_free).  Returns the number of slices. */
int amgb_sellu_encode_host(int nrows, const int *row_ptr, const int *col_idx, const double *values, const double *scaled_values,
                           int **slice_desc, int **delta, unsigned int **mask, double **gvalues, double **gscaled, int *ngroups);
void amgb_host_free(void *p);
/* coarse-hierarchy bytes living in the L2-pinned arena (cudaAccessPolicyWindow of the persistent kernel) */
int amgb_l2_arena_bytes(amgb_ctx *ctx, long long *used, long long *capacity);

/* ---- multi-GPU (DMEM replacement; one process per GPU) ------------------------------------
 * Replaces DMEM_Add / DMEM_SyncAdd (src/DMEM_Add.cpp:20-178, src/DMEM_Mult.cpp:263-450) for the synchronous
 * Multadd and BPX cycles, and AFACx with the SMEM meaning (src/SEQ_AMG.cpp:172-208), with weighted or L1 Jacobi, one sweep per level: hypre's ParCSR halo exchange and DMEM_Comm (src/DMEM_Comm.cpp:81-382) become NCCL
 * send/recv between row-neighbours, the residual norm an ncclAllReduce (src/DMEM_Misc.cpp:398-433).
 * Call order: amgb_create, amgb_dist_init, amgb_set_options, amgb_set_num_levels, amgb_dist_set_level for
 * EVERY level, then the amgb_set_matrix calls (LOCAL row blocks whose column
 * indices are in the rank's extended numbering [ghost_lo | owned | ghost_hi] on distributed levels, full
 * matrices on replicated levels), amgb_setup, amgb_dist_setup. */
/* rank 0 obtains a 128-byte NCCL unique id and distributes it (MPI_Bcast / torch.distributed broadcast) */
int amgb_dist_unique_id(unsigned char id128[128]);
int amgb_dist_init(amgb_ctx *ctx, const unsigned char id128[128], int rank, int nranks);
/* vector layout of one level on this rank: owned rows [row_start, row_start + n_owned) of n_global;
 * distributed != 0: halo_lo / halo_hi ghost entries come from rank-1 / rank+1, and this rank sends its
 * first send_lo / last send_hi owned entries to them; distributed == 0: the level is replicated (full
 * vectors, redundant computation), row_start / n_owned then name the slice this rank contributes to the
 * all-gather of the first replicated level.  all_owned[nranks] = n_owned of every rank. */
int amgb_dist_set_level(amgb_ctx *ctx, int level, int n_global, int row_start, int n_owned, int halo_lo, int halo_hi,
                        int distributed, int send_lo, int send_hi, const int *all_owned);
int amgb_dist_setup(amgb_ctx *ctx);
int amgb_dist_set_rhs(amgb_ctx *ctx, const double *f_owned);        /* this rank's rows of f */
int amgb_dist_get_solution(amgb_ctx *ctx, double *u_owned);
/* x0 = 0; cycles until ||r||/||r0|| < tol (global norms) or max_cycles; identical history on every rank */
int amgb_dist_solve_sync(amgb_ctx *ctx, double tol, int max_cycles, double *relres_hist, int *n_cycles,
                         double *solve_seconds);
/* the same with DMEM's acceleration of the accumulated correction (DMEM_ChebyUpdate, src/DMEM_Misc.cpp:612-666, applied in
 * DMEM_SyncAddCorrect src/DMEM_Add.cpp:706-711): accel 0 none, 1 Chebyshev, 2 second-order Richardson; mu, delta from
 * ChebySetup (src/DMEM_Setup.cpp:1901-1914) */
int amgb_dist_solve_sync_accel(amgb_ctx *ctx, double tol, int max_cycles, int accel, double mu, double delta,
                               double *relres_hist, int *n_cycles, double *solve_seconds);
/* DMEM_PowerMult (src/DMEM_Eig.cpp:10-104): extreme eigenvalues of B*A by `iters` steps of power iteration (second, deflated pass
 * for the minimum) on the partitioned path, B = this context's additive cycle from a zero guess; u0_owned = this rank's rows of
 * the start vector (the reference: RandDouble(0,1) - .5 after srand(rank)), NULL = all ones.  Collective: every rank calls it and
 * receives the same bounds; DMEM's ChebySetup takes alpha = eig_min, beta = eig_max (src/DMEM_Setup.cpp:1901-1914). */
int amgb_dist_eigs_power(amgb_ctx *ctx, int iters, const double *u0_owned, double *eig_min, double *eig_max);
int amgb_dist_stats(amgb_ctx *ctx, long long *halo_bytes_sent, long long *nccl_ops);

/* ---- asynchronous additive solve, ROW-PARTITIONED over the GPUs: DMEM_Add's asynchronous loop (src/DMEM_Add.cpp:101-130)
 * with DMEM_AddCorrect_LocalRes / DMEM_AddResidual_LocalRes (:391-556) and DMEM_Comm's Isend / Test engine
 * (src/DMEM_Comm.cpp:81-382).  On a context prepared with amgb_dist_init .. amgb_dist_setup (Multadd or AFACx, weighted / L1
 * Jacobi) every rank runs ONE persistent kernel on its row blocks: the level groups loop over the single-GPU programs and
 * store the boundary entries of every vector a later SpMV reads with ghosts straight into the neighbour GPUs' ghost slots
 * (CUDA IPC over NVLink; the handles and layouts travel through NCCL all-gathers inside the first call); nobody waits for
 * a peer.  From the resident f and u; LOCAL stop rule: every group of every rank performs num_cycles corrections.
 * Collective.  corrections[num_levels]: this rank's counts; relres = global ||f - A u|| / ||f - A u_start||; solve_seconds =
 * this rank's kernel time (the job's time is the maximum over the ranks). */
int amgb_dist_solve_async(amgb_ctx *ctx, int num_cycles, int *corrections, double *relres, double *solve_seconds);
int amgb_dist_async_groups(amgb_ctx *ctx, int *cta_begin /* num_levels + 1 */, double *group_seconds /* num_levels */);
/* host-only probe (no CUDA call) of the planning behind amgb_dist_solve_async, for the CPU test suite's multi-rank
 * interpreter: layouts = nranks x num_levels x 8 ints (n_global, row_start, n_owned, halo_lo, halo_hi, distributed, send_lo,
 * send_hi); ops = max_ops records of csrc/launch.h DistAsyncOp; a vector is a slot of the rank's arena, slot_off in doubles */
int amgb_dist_async_plan(const amgb_options *opt, int num_levels, int nranks, int rank, const int *layouts, int symmetric,
                         int factor_level0, void *ops, int max_ops, int *op_begin, long long *slot_off, int *slot_group,
                         int *slot_vec, int max_slots, int *num_slots);

/* ---- asynchronous fine-grid smoother across GPUs: DMEM_AsyncSmooth (src/DMEM_Smooth.cpp:16-313) with the ASYNC_JACOBI /
 * ASYNC_L1_JACOBI smoothers, the `-smoother async_j` solver of DMEM_Add (src/DMEM_Add.cpp:88-95).  Every rank relaxes its
 * rows of A_0 x = f again and again, x_own += s o (f - A_0 [ghosts | x_own]), with whatever ghost values have arrived, and
 * writes its new boundary entries straight into the neighbours' ghost slots (their level-0 vectors mapped through CUDA IPC:
 * stores over NVLink replace finestIntra_outsideSend / Recv and DMEM_Comm's Isend / Test engine).  Nobody waits.
 * amgb_dist_ipc_export_solution: 64-byte handle of this rank's level-0 vector.  amgb_dist_ipc_open_neighbours: the handles
 * of rank-1 / rank+1 (NULL where there is none); lo_ghost_offset = rank-1's halo_lo + n_owned (index of its first ghost_hi
 * entry).  amgb_dist_async_smooth enqueues `sweeps` relaxations (LOCAL stop rule, AsyncSmoothCheckConverge :340-349) and
 * returns without synchronising.  amgb_dist_residual_norm: global ||f - A_0 x||_2 (collective; synchronises). */
int amgb_dist_ipc_export_solution(amgb_ctx *ctx, unsigned char handle64[64]);
int amgb_dist_ipc_open_neighbours(amgb_ctx *ctx, const unsigned char *handle_lo, long long lo_ghost_offset,
                                  const unsigned char *handle_hi);
int amgb_dist_async_smooth(amgb_ctx *ctx, int sweeps);
int amgb_dist_residual_norm(amgb_ctx *ctx, double *norm);
int amgb_dist_zero_solution(amgb_ctx *ctx);

/* ---- asynchronous additive solve across GPUs (DMEM async Multadd; one process per GPU) --------------------------
 * The reference assigns ranks to grids (src/DMEM_Setup.cpp:1638-1759): every grid's rank group holds the hierarchy
 * down to its level and full-length fine vectors, runs its own chain on a private residual and sends fine-level
 * corrections to the other grids, which accumulate them on arrival (src/DMEM_Add.cpp:101-130,391-458;
 * src/DMEM_Comm.cpp:267-330).  Here a GPU plays a grid's rank group; every context holds the whole hierarchy
 * (amgb_set_matrix as for one GPU) and the same f.  amgb_ipc_export_solution / amgb_ipc_open_peers map the peers'
 * solution vectors through CUDA IPC; amgb_async_dist_correct(level) enqueues ONE correction of `level`: private copy
 * of u, r = f - A_0 u, restrict chain, smooth, prolong chain, then u += e on this GPU and on every peer with fp64
 * reductions over NVLink.  No call ever waits for a peer.  amgb_residual_norm = ||f - A_0 u||_2 (synchronises the
 * context's stream). */
int amgb_ipc_export_solution(amgb_ctx *ctx, unsigned char handle64[64]);
int amgb_ipc_open_peers(amgb_ctx *ctx, int npeers, const unsigned char *handles /* npeers x 64 bytes */);
int amgb_async_dist_correct(amgb_ctx *ctx, int level);
int amgb_residual_norm(amgb_ctx *ctx, double *norm);
int amgb_stream_synchronize(amgb_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif

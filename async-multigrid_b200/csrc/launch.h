// launch.h -- host-side launchers of the stand-alone kernels (kernels.cu) and of the persistent
// asynchronous kernel (async.cu).  Every launcher returns the number of kernels it launched.
#pragma once
#include "common.cuh"
#include "amg_b200.h"
#include <vector>

struct LaunchCfg {
   int num_sms = 148;
   int ctas_per_sm = 8;
   int stream_variant = 0;
   int sellu_ctas = 5;          // SELL-U kernel variant (AMGB_SELLU_CTAS): cached-delta path at 5 (48 registers, default), 4 (64) or 6 (40, spills)
                                // CTAs per SM; 8 = the generic batch-of-8 loop at 4 CTAs per SM (56 registers)
};

// geometry of the CSR-stream kernel (kernels.cuh stream_rows_team): threads per CTA, entries per row block,
// staged-x window capacity (0 = gather x from global memory), bulk-copy stages.  amgb_options.stream_variant
// selects one; the row blocks are built for its cap / xcap at upload time.
struct StreamVariant { int nt, cap, xcap, stages; };
// stages == 0: the warp-granular variant (warp_stream_rows_team), cap = entries per warp chunk
// stages == -1: warp-granular with column-sorted chunks (DevCSR::pci/pva/pos)
#define AMGB_NUM_STREAM_VARIANTS 13
static const StreamVariant kStreamVariants[AMGB_NUM_STREAM_VARIANTS] = {
   {256, 2048, 0, 3}, {128, 1024, 0, 2}, {128, 1024, 0, 3}, {256, 2048, 1536, 2},
   {128, 1024, 1024, 2}, {256, 1024, 0, 2}, {128, 1024, 1024, 3}, {128, 2048, 0, 2},
   {256, 256, 0, 0}, {256, 128, 0, 0}, {256, 512, 0, 0}, {256, 256, 0, -1}, {256, 128, 0, -1},
};

// y = gamma*c + rs.*(beta*b + alpha*M*x); optional sum of y_i^2 -- or of y_i*dot_w_i when dot_w is given -- into partial
// sums (one per CTA, `partials` must hold >= grid entries; *grid_out receives the grid used).
int launch_spmv(const LaunchCfg &cfg, cudaStream_t st, const DevCSR &M, bool use_sval, const double *x, double *y,
                const SpmvEpilogue &e, double *partials, int *grid_out, const double *dot_w = nullptr);
int spmv_units(const DevCSR &M);
int launch_spmv_units(const LaunchCfg &cfg, cudaStream_t st, const DevCSR &M, int u0, int u1, bool use_sval, const double *x,
                      double *y, const SpmvEpilogue &e, double *partials, int *grid_out, const double *dot_w = nullptr);
// out[0] = sum(partials[0..n)); if hist != nullptr: hist[k] = sqrt(out[0]) (and r0 handling on host)
int launch_reduce_partials(cudaStream_t st, const double *partials, int n, double *out);
// y = a.*x  (zero-guess Jacobi: u = (w/d).*f, src/SMEM_Smooth.cpp:381-389)
int launch_scale(const LaunchCfg &cfg, cudaStream_t st, int n, const double *a, const double *x, double *y);
// y += x
int launch_add(const LaunchCfg &cfg, cudaStream_t st, int n, const double *x, double *y);
// Chebyshev update (src/SMEM_Solve.cpp:179-187): uo_prev=uo; uo = yo + omega*(delta*c + uo - yo); yo = uo_prev; u = uo
int launch_cheby(const LaunchCfg &cfg, cudaStream_t st, int n, double omega, double delta, const double *c,
                 double *u_outer, double *y_outer, double *u);
// y = a*x + b*y [, z = y]; partial sums of x_i*y_i
int launch_axpby(const LaunchCfg &cfg, cudaStream_t st, int n, double a, const double *x, double b, double *y, double *z);
int launch_dot(const LaunchCfg &cfg, cudaStream_t st, int n, const double *x, const double *y, double *partials, int *grid_out);
// preconditioned conjugate gradients (pcg.cu): slots of the device scalar array.  Each reduction writes its own slot;
// k_pcg_update records rho_old and the number of completed iterations (0 = the next direction is the first)
enum { PCG_RHO = 0, PCG_SIGMA = 1, PCG_RR = 2, PCG_RHO_OLD = 3, PCG_DONE = 4, PCG_NSCALARS = 8 };
// p = z + beta p with beta from s (p = z on the first iteration)
int launch_pcg_dir(const LaunchCfg &cfg, cudaStream_t st, int n, const double *z, double *p, const double *s);
// alpha = rho / sigma from s; u += alpha p; r -= alpha q (skipped on a breakdown); partial sums of r_i^2
int launch_pcg_update(const LaunchCfg &cfg, cudaStream_t st, int n, const double *p, const double *q, double *u, double *r,
                      double *s, double *partials, int *grid_out);
// u += e here and on every peer GPU (IPC-mapped pointers)
#define AMGB_MAX_PEERS 15
struct PeerPtrs { double *p[AMGB_MAX_PEERS]; int n; };
int launch_push_correction(const LaunchCfg &cfg, cudaStream_t st, int n, const double *e, double *u, const PeerPtrs &peers);
// partial sums of x_i^2
int launch_sumsq(const LaunchCfg &cfg, cudaStream_t st, int n, const double *x, double *partials, int *grid_out);
// hybrid JGS sweep
int launch_hybrid_jgs(const LaunchCfg &cfg, cudaStream_t st, const DevCSR &A, const double *f, double *u,
                      const double *u_prev, const double *scale, int block_rows, bool zero_guess);
// the same sweep over an explicit block list bounds[0..nblocks] (amgb_set_jgs_blocks: the reference's blocks are thread row ranges)
int launch_hybrid_jgs_list(const LaunchCfg &cfg, cudaStream_t st, const DevCSR &A, const double *f, double *u,
                           const double *u_prev, const double *scale, const int *bounds, int nblocks, bool zero_guess);
// (semi-)asynchronous Gauss-Seidel sweeps on u (in place); y = M^T x
int launch_async_gs(const LaunchCfg &cfg, cudaStream_t st, const DevCSR &A, const double *f, double *u, int block_rows,
                    int sweeps, bool semi);
int launch_spmv_transpose(const LaunchCfg &cfg, cudaStream_t st, const DevCSR &M, const double *x, double *y);
// setup helpers: ws = w/d (0 where d == 0), l1 = sum |a_ij|, sval = va .* cs[col]
int launch_diag_scale(cudaStream_t st, const DevCSR &A, double w, double *ws, double *dow);
int launch_l1(cudaStream_t st, const DevCSR &A, double *l1, double *inv_l1);
int launch_diag_scale_vec(cudaStream_t st, int n, const double *diag, const double *l1src, double w, double *ws, double *dow,
                          double *l1, double *inv_l1);
int launch_colscale(cudaStream_t st, int nnz, const int *ci, const double *va, const double *cs, double *out);

// ---- persistent asynchronous kernel (async.cu) ---------------------------------------------------
// The kernel is an interpreter: every level's CTA group loops over its own PROGRAM, a short list of operations (SpMV with a
// fused epilogue, vector ops, smoother sweeps, the correction count / stop test) separated by group barriers.  The host
// builds the programs from the solver options (async_build_program, pure host code: the CPU test suite interprets the same
// programs in numpy against the CPU restatement), so Multadd / AFACx, explicit or factorised level-0 transfers, -read_type,
// -res_compute_type and -async_type are host-side variations of one small kernel.
#define AMGB_MAX_LEVELS 32
enum { AOP_SPMV = 0, AOP_SCALE = 1, AOP_COPY = 2, AOP_ZERO = 3, AOP_UPDATE = 4, AOP_COUNT_STOP = 5, AOP_LOCK = 6, AOP_UNLOCK = 7,
       AOP_JGS = 8, AOP_ASYNC_GS = 9,
       // row-partitioned solve (dist_async.cu): PUSH = boundary / owned entries of a vector into a peer GPU's ghost slots;
       // SIGNAL = "this group's stores of exchange step s are in place" into a peer's flag word; WAIT = until a peer's flag says s
       AOP_PUSH = 10, AOP_SIGNAL = 11, AOP_WAIT = 12,
       // asynchronous implicit extended-system BPX (extended.cu; the EXT instantiation of the kernel only):
       // EXT_RESID = an SpMV like AOP_SPMV whose rows' sum of squares goes into this CTA's slot AsyncExtParams::cta_ss;
       // EXT_CHEBY = y <- c + omega (delta rs o x + y - c), c <- old y over level `level` (x = r_k, y = u_k, c = y_k), then
       //             omega <- 1 / (1 - omega / (2 mu)^2) in every CTA of the group; EXT_STOP = the group's count / stop rule
       AOP_EXT_RESID = 13, AOP_EXT_CHEBY = 14, AOP_EXT_STOP = 15 };
// vectors a program names: id = kind * 64 + level (group-private unless said otherwise)
enum { AV_NONE = -1, AV_F = 0 /* shared f */, AV_U = 1 /* shared u */, AV_RS = 2 /* shared residual (GLOBAL / READ_RES) */,
       AV_R = 3, AV_E = 4, AV_T = 5, AV_W = 6, AV_UL = 7 /* private copy of u */, AV_T0 = 8 /* level-0 scratch */,
       AV_FACC = 9 /* accumulated corrections (READ_RES) */, AV_WS = 10 /* w/d (read-only) */, AV_INVL1 = 11 /* 1/l1 (read-only) */,
       // extended-system programs: the shared per-level vectors f_l, u_l, y_l, e_l (ExtState), and the group-private chain
       // vectors z1_l (prolongation chain), z2_l (restriction chain; z2_l + e_l on the levels the chain passes) and r_l
       AV_XF = 12, AV_XU = 13, AV_XY = 14, AV_XE = 15, AV_XZ1 = 16, AV_XZ2 = 17, AV_XR = 18 };
#define AV_ID(kind, level) ((kind) * 64 + (level))
#define AMAT_AINV 3                // AsyncOp::mat_kind beside AMGB_MAT_A / P / R: the dense inverse of the coarsest operator (coarse_solve)
struct AsyncOpSym {                // one operation, symbolic (what the CPU tests interpret)
   int type;                       // AOP_*
   int mat_kind, mat_level;        // AOP_SPMV / AOP_JGS / AOP_ASYNC_GS: AMGB_MAT_* and level
   int sval;                       // AOP_SPMV: the column-scaled values A*diag(w/d)
   int range;                      // 0: the whole operation is shared by the CTAs of the group; 1: this CTA's slice of the level-0 rows
                                   //    (rows dealt to ALL CTAs of the grid: -res_compute_type global)
   int barrier;                    // group barrier after the operation
   int x, y;                       // input / output vector ids (y = AV_NONE: the result goes to the reduction target only)
   int b, c, rs, b2, xs;           // epilogue operands: y_i = gamma*c_i + rs_i*(beta*b_i + beta2*b2_i + alpha*(M x)_i) + xself*xs_i
   int red, red_copy, acc;         // red += red_scale * y_i (fp64 reduction into a SHARED vector), red_copy_i = red_i afterwards; acc_i += y_i
   int level, sweeps, zero;        // smoother operations: level, sweeps, zero initial guess
   int locked;                     // AOP_UPDATE: plain read-modify-write (inside the SEMI_ASYNC critical section) instead of reductions
   double alpha, beta, gamma, beta2, xself, red_scale;
};
struct AsyncOp {                   // the same with device pointers (AOP_PUSH: `sweeps` doubles from x to y, y in a peer's memory;
                                   // AOP_SIGNAL: y = the peer's flag word, zero = first signal of an exchange step; AOP_WAIT: x = own flag word)
   int type, mat_kind, mat_level, sval, range, barrier, level, sweeps, zero, locked;
   const double *x;
   double *y;
   SpmvEpilogue e;
};
struct AsyncParams {
   int num_levels;
   int first_group;                // 0; 1 with -res_compute_type global (level 0 has no group of its own)
   int smoother;
   int jgs_block_rows;
   int jgs_lpb[AMGB_MAX_LEVELS];  // lanes per hybrid-JGS block on every level (4/8/16/32 from the mean row length; 0: one thread per block)
   int num_cycles;
   int converge_type;
   DevCSR A[AMGB_MAX_LEVELS], P[AMGB_MAX_LEVELS], R[AMGB_MAX_LEVELS];
   DevCSR Ainv;                             // coarse_solve: A_{L-1}^{-1} as a full CSR
   int cta_begin[AMGB_MAX_LEVELS + 1];      // CTA range of every level's group
   int slice_ctas;                          // CTAs that share the level-0 rows of the CTA-slice operations (the working groups')
   const AsyncOp *ops;                      // all programs, group after group
   int op_begin[AMGB_MAX_LEVELS + 1];       // program of group q: ops[op_begin[q] .. op_begin[q+1])
   int n0;
   double *u;                               // shared fine solution
   unsigned int *barrier_count;             // [L] arrive counters
   volatile unsigned int *barrier_gen;      // [L] generations
   int *num_correct;                        // [L] local_num_correct
   int *group_stop;                         // [L] the group root's stop decision (GLOBAL rule)
   volatile int *converge_flag;             // thread.converge_flag
   int *lock;                               // SEMI_ASYNC: the omp lock around "u += e; u_k = u"
   unsigned long long *group_ns;            // [L] nanoseconds every group spent in the kernel (CTA-group balancing)
   // asynchronous implicit extended-system BPX only (the EXT instantiation reads these; the others never do)
   struct AsyncExtParams {
      double delta, mu22;                   // Chebyshev: delta, (2 mu)^2
      double tol, r0_ext;                   // stop when sqrt(sum of the published contributions) / r0_ext < tol
      double *cta_ss;                       // [grid] sum of r^2 over this CTA's rows of its group's last residual
      volatile double *contrib;             // [L] published sum r_k^2 of every group (1e300 = not measured yet)
      int *loc_iters;                       // [L] every group's loc_iters at exit
      int *done;                            // groups whose loc_iters reached num_cycles
   } ext;
};
// heavy: the instantiation that carries the Gauss-Seidel-type smoothers (more registers, fewer CTAs per SM)
int launch_async(cudaStream_t st, const AsyncParams *params_dev, int grid, int block, bool heavy, const cudaAccessPolicyWindow *window);
int async_max_grid(int block, bool heavy);
// the instantiation that carries the extended-system operations (AOP_EXT_*)
int launch_async_ext(cudaStream_t st, const AsyncParams *params_dev, int grid, int block, const cudaAccessPolicyWindow *window);
int async_max_grid_ext(int block);
// host-only: the program of group q (appended to `ops`); returns AMGB_OK or AMGB_EINVAL for an unsupported combination
int async_build_program(const amgb_options &o, int L, bool symmetric, bool fact0, int q, std::vector<AsyncOpSym> &ops, bool partitioned = false);
// host-only: the program of group q of the asynchronous implicit extended-system solver (appended to `ops`); AMGB_EINVAL for
// smoothers other than weighted / L1 Jacobi
int async_build_ext_program(const amgb_options &o, int L, int q, std::vector<AsyncOpSym> &ops);
// CTA groups in proportion to `work` (at least one CTA per group from `first` on): cta_begin[L + 1]
void async_deal_ctas(const std::vector<double> &work, int L, int first, int grid, int *cta_begin);

// ---- row-partitioned asynchronous solve (dist_async.cu): the same programs on every GPU's row blocks, with AOP_PUSH
// operations after every operation whose result a later SpMV reads with ghosts.  Pure host planning, shared by the device
// path and the CPU test suite's multi-rank interpreter: vectors are SLOTS of one arena per rank (identical slot table on
// every rank, a slot holds the largest extended length over the ranks), an operand is (slot, element offset).
struct DistLay { int n_global, row_start, n_owned, halo_lo, halo_hi, distributed, send_lo, send_hi; };   // one (rank, level)
enum { DROLE_X = 0, DROLE_Y, DROLE_B, DROLE_C, DROLE_RS, DROLE_B2, DROLE_XS, DROLE_RED, DROLE_RED_COPY, DROLE_ACC, DROLE_N };
enum { DEXT_NONE = -1, DEXT_F = -2 /* rhs, owned rows */, DEXT_U = -3 /* shared solution, level-0 layout */,
       DEXT_WS0 = -100 /* DEXT_WS0 - l: w/d or 1/l1 of level l, level layout */ };
struct DistAsyncOp {
   int type, mat_kind, mat_level, sval, barrier, level;
   int count, dst_rank;             // AOP_PUSH: `count` doubles from (slot[X], elem[X]) here to (slot[Y], elem[Y]) on dst_rank (-1: nobody there);
                                    // AOP_SIGNAL: to dst_rank, count = 1 on the first signal of an exchange step; AOP_WAIT: for dst_rank
   int slot[DROLE_N];               // >= 0: arena slot; DEXT_*
   long long elem[DROLE_N];         // first element of the operand inside the slot / external vector
   double alpha, beta, gamma, beta2, xself, red_scale;
};
struct DistAsyncPlan {
   std::vector<DistAsyncOp> ops;           // all groups, group after group
   std::vector<int> op_begin;              // [L + 1]
   std::vector<long long> slot_off;        // [num_slots + 1], doubles
   std::vector<int> slot_group, slot_vec;  // which group's which vector (AV_ID) a slot holds
   // after the last slot: L x nranks 8-byte flag words, flag[q * nranks + src] = last exchange step of group q that rank src
   // has completed towards this rank (slot_off.back() is where they start)
};
// lay[p * L + l]; returns AMGB_OK or AMGB_EINVAL (unsupported options / inconsistent layouts)
int dist_async_plan(const amgb_options &o, int L, int nranks, int rank, const DistLay *lay, bool symmetric, bool fact0, DistAsyncPlan &out);

// extended.cu -- implicit extended-system BPX solver (`-solver iebpx`) on the device.
//
// Replaces SMEM_ExtendedSystemSolve with IMPLICIT_EXTENDED_SYSTEM_BPX (src/SMEM_ExtendedSystem.cpp:9-836, finish :777-817,
// ExtendedSystemImplicitMatVec :838-907): Chebyshev-accelerated Jacobi on Griebel's semi-definite generating system whose
// unknowns are the per-level vectors u_0 .. u_{L-1}; block (k,l) of the operator is A_k P^{k<-l} for l >= k and
// R^{k<-l} A_l for l < k and is never formed.  Plain P, R = P^T (src/SMEM_Setup.cpp:262-274).
//
//   set-up      f_{l+1} = R_l f_l;  r0_ext = sqrt(sum_l |f_l|^2);  y_l = 0;  u_l = delta f_l ./ diag(A_l);  e_l = A_l u_l
//   iteration   phase 1 (all levels, from the same u, e):   z1_{L-1} = u_{L-1},  z1_k = P_k z1_{k+1} + u_k
//                                                           z2_0 = 0,           z2_{k+1} = R_k (z2_k + e_k)
//               phase 2 (level k):  r_k = f_k - (A_k z1_k + z2_k);  s = r_k ./ scale_k  (a_ii/w or the L1 norm)
//                                   u_k <- y_k + omega (delta s + u_k - y_k),  y_k <- old u_k;  e_k = A_k u_k
//               omega <- 1 / (1 - omega/(2 mu)^2)
//   finish      extended residual of the final iterate;  x = sum_l P^{0<-l} u_l;  r = f - A_0 x
//
// The reference gives every level a thread group that recomputes the z1 / z2 chains it needs (level k: L-1-k prolongations
// and k restrictions, sum over k = L(L-1) SpMVs per iteration); the chains are the same for all groups, so here they are
// computed once per iteration (2(L-1) SpMVs) and shared.  Everything is a composition of the kernels of kernels.cuh: the
// prolongation fuses "+ u_k", the residual fuses "f_k - z2_k - A_k z1_k" and its sum of squares.
//
// The EXPLICIT form (`-solver eebpx`, EXPLICIT_EXTENDED_SYSTEM_BPX, :84-110,295-365) is the same loop on a ONE-level
// context whose A_0 is the assembled extended matrix AA (BuildExtendedMatrix, src/SMEM_Setup.cpp:1426-1521; host side:
// amgh_build_extended_matrix) with smooth_weight = 1 (that branch divides by the raw diagonal): z1 = x, z2 = 0,
// r = bb - AA x, x <- y + omega (delta r ./ diag + x - y).  solver.ExtendedExplicitSolver drives it.
#include "ctx.h"
#include "async_team.cuh"
#include <algorithm>
#include <cmath>
#include <cstring>

struct ExtState {
   std::vector<double *> f, u, y, e, z1, z2, s, r, us;
   // asynchronous implicit form (amgb_solve_extended_implicit_async), prepared at its first call: the parameter block of the
   // persistent kernel (programs resolved to device pointers, CTA groups, counters), its device copy and the L2 window
   bool async_ready = false;
   AsyncParams hp;
   void *params_dev = nullptr;
   cudaAccessPolicyWindow window = {};
};

void amgb_ext_teardown(amgb_ctx *c)
{
   delete c->ext;
   c->ext = nullptr;
}

static inline SpmvEpilogue epi(double alpha, double beta, const double *b, double gamma = 0.0, const double *cc = nullptr,
                               const double *rs = nullptr)
{
   SpmvEpilogue e;
   e.alpha = alpha; e.beta = beta; e.gamma = gamma; e.b = b; e.c = cc; e.rs = rs;
   return e;
}

static int ext_alloc(amgb_ctx *c)
{
   if (c->ext) return AMGB_OK;
   ExtState *x = new ExtState();
   const int L = c->L;
   std::vector<double *> *arrs[] = {&x->f, &x->u, &x->y, &x->e, &x->z1, &x->z2, &x->s, &x->r, &x->us};
   for (auto a : arrs) {
      a->assign(L, nullptr);
      for (int l = 0; l < L; l++) {
         int rc = amgb_dev_alloc_bytes(c, (void **)&(*a)[l], sizeof(double) * (size_t)std::max(1, c->A[l].nrows), true);
         if (rc) { delete x; return rc; }
      }
   }
   c->ext = x;
   return AMGB_OK;
}

// z1 / z2 chains from the current u, e (phase 1; also the first half of ExtendedSystemImplicitMatVec)
static void ext_phase1(amgb_ctx *c, ExtState *x)
{
   const int L = c->L;
   cudaMemcpyAsync(x->z1[L - 1], x->u[L - 1], sizeof(double) * (size_t)c->A[L - 1].nrows, cudaMemcpyDeviceToDevice, c->stream);
   for (int k = L - 2; k >= 0; k--) enq_spmv(c, c->P[k], false, x->z1[k + 1], x->z1[k], epi(1.0, 1.0, x->u[k]), false);
   // z2_0 stays zero (allocated zeroed, never written)
   for (int k = 0; k < L - 1; k++) {
      const double *in = x->e[k];
      if (k > 0) {   // s_k = z2_k + e_k: z2_k itself is still needed by phase 2
         cudaMemcpyAsync(x->s[k], x->z2[k], sizeof(double) * (size_t)c->A[k].nrows, cudaMemcpyDeviceToDevice, c->stream);
         c->launches += launch_add(c->cfg, c->stream, c->A[k].nrows, x->e[k], x->s[k]);
         in = x->s[k];
      }
      enq_spmv(c, c->R[k], false, in, x->z2[k + 1], epi(1.0, 0.0, nullptr), false);
   }
}

// r_k = f_k - z2_k - A_k z1_k for every level, d_scalars[1 + k] = |r_k|^2
static void ext_residuals(amgb_ctx *c, ExtState *x)
{
   for (int k = 0; k < c->L; k++) {
      SpmvEpilogue e = epi(-1.0, 1.0, x->f[k]);
      e.b2 = x->z2[k]; e.beta2 = -1.0;
      int grid = 0;
      c->launches += launch_spmv(c->cfg, c->stream, c->A[k], false, x->z1[k], x->r[k], e, c->partials, &grid);
      c->launches += launch_reduce_partials(c->stream, c->partials, grid, c->d_scalars + 1 + k);
   }
}

static int ext_fetch_sum(amgb_ctx *c, double *out)
{
   const int L = c->L;
   CUDA_OK(c, cudaMemcpyAsync(c->h_scalars + 1, c->d_scalars + 1, sizeof(double) * (size_t)L, cudaMemcpyDeviceToHost, c->stream));
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   double s = 0.0;
   for (int k = 0; k < L; k++) s += c->h_scalars[1 + k];
   *out = s;
   return AMGB_OK;
}

// set-up shared by the synchronous and the asynchronous implicit solver (src/SMEM_ExtendedSystem.cpp:112-136):
// f_{l+1} = R_l f_l;  r0 = |f|, r0_ext = sqrt(sum_l |f_l|^2);  y_l = 0;  u_l = delta f_l ./ a_ii;  e_l = A_l u_l
static int ext_setup(amgb_ctx *c, ExtState *x, double delta, double *r0, double *r0_ext)
{
   const int L = c->L, n0 = c->A[0].nrows;
   int rc, grid = 0;
   CUDA_OK(c, cudaMemcpyAsync(x->f[0], c->f, sizeof(double) * (size_t)n0, cudaMemcpyDeviceToDevice, c->stream));
   for (int l = 0; l < L - 1; l++) enq_spmv(c, c->R[l], false, x->f[l], x->f[l + 1], epi(1.0, 0.0, nullptr), false);
   for (int l = 0; l < L; l++) {
      c->launches += launch_sumsq(c->cfg, c->stream, c->A[l].nrows, x->f[l], c->partials, &grid);
      c->launches += launch_reduce_partials(c->stream, c->partials, grid, c->d_scalars + 1 + l);
   }
   double ss;
   if ((rc = ext_fetch_sum(c, &ss))) return rc;
   *r0 = sqrt(c->h_scalars[1]);
   *r0_ext = sqrt(ss);
   for (int l = 0; l < L; l++) {
      const int n = c->A[l].nrows;
      CUDA_OK(c, cudaMemsetAsync(x->y[l], 0, sizeof(double) * (size_t)n, c->stream));
      // u = delta f ./ a_ii: ws = w/d, so f .* ws scaled by delta/w
      c->launches += launch_scale(c->cfg, c->stream, n, c->ws[l], x->f[l], x->u[l]);
      c->launches += launch_axpby(c->cfg, c->stream, n, 0.0, x->f[l], delta / c->opt.smooth_weight, x->u[l], nullptr);
      if (L > 1) enq_spmv(c, c->A[l], false, x->u[l], x->e[l], epi(1.0, 0.0, nullptr), false);   // e feeds the restriction chain only
   }
   return AMGB_OK;
}

// finish shared by both implicit solvers (:777-817): extended residual of the final u_l, then x = sum_l P^{0<-l} u_l into u
static int ext_finish(amgb_ctx *c, ExtState *x, double r0_ext, double *ext_relres)
{
   const int L = c->L, n0 = c->A[0].nrows;
   int rc;
   double ss;
   ext_phase1(c, x);
   ext_residuals(c, x);
   if ((rc = ext_fetch_sum(c, &ss))) return rc;
   if (ext_relres) *ext_relres = sqrt(ss) / r0_ext;
   for (int k = L - 2; k >= 0; k--) {
      // u_k += P_k u_{k+1}  (out of place through s_k: the kernel must not write the vector other rows' epilogues read)
      enq_spmv(c, c->P[k], false, x->u[k + 1], x->s[k], epi(1.0, 1.0, x->u[k]), false);
      CUDA_OK(c, cudaMemcpyAsync(x->u[k], x->s[k], sizeof(double) * (size_t)c->A[k].nrows, cudaMemcpyDeviceToDevice, c->stream));
   }
   CUDA_OK(c, cudaMemcpyAsync(c->u, x->u[0], sizeof(double) * (size_t)n0, cudaMemcpyDeviceToDevice, c->stream));
   return AMGB_OK;
}

// the checks both implicit solvers make before any work
static int ext_check(amgb_ctx *c, int num_cycles, double mu)
{
   if (c->L + 1 > 64) return amgb_fail(c, AMGB_EINVAL, "too many levels");
   if (num_cycles < 0 || mu == 0.0) return amgb_fail(c, AMGB_EINVAL, "bad arguments");
   if (c->dist) return amgb_fail(c, AMGB_EINVAL, "the extended-system solver runs on one GPU");
   const int sm = c->opt.smoother;
   if (sm != AMGB_SMOOTH_JACOBI && sm != AMGB_SMOOTH_L1_JACOBI)
      return amgb_fail(c, AMGB_EINVAL, "the extended-system solver runs with weighted or L1 Jacobi");
   if (c->opt.solver != AMGB_SOLVER_BPX && c->opt.solver != AMGB_SOLVER_IEBPX)
      return amgb_fail(c, AMGB_EINVAL, "the extended-system solver needs the plain transfers of BPX (solver BPX or IEBPX)");
   return AMGB_OK;
}

extern "C" int amgb_solve_extended(amgb_ctx *c, double tol, int num_cycles, double mu, double delta, double *ext_hist, int *iters,
                                   double *ext_relres, double *relres, double *solve_seconds)
{
   NEED_READY(c);
   const int L = c->L;
   int rc;
   if ((rc = ext_check(c, num_cycles, mu))) return rc;
   const int sm = c->opt.smoother;
   if ((rc = ext_alloc(c))) return rc;
   ExtState *x = c->ext;
   double r0, r0_ext, ss;
   if ((rc = ext_setup(c, x, delta, &r0, &r0_ext))) return rc;
   double omega = 2.0;
   const double mu22 = (2.0 * mu) * (2.0 * mu);
   int it = 1;
   CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
   if (num_cycles > 1)
      for (;;) {
         ext_phase1(c, x);
         ext_residuals(c, x);
         for (int k = 0; k < L; k++) {
            const int n = c->A[k].nrows;
            const double *rs = (sm == AMGB_SMOOTH_L1_JACOBI) ? c->inv_l1[k] : c->ws[k];
            c->launches += launch_scale(c->cfg, c->stream, n, rs, x->r[k], x->us[k]);
            // u <- y + omega (delta s + u - y), y <- old u   (k_cheby; its third output goes to scratch)
            c->launches += launch_cheby(c->cfg, c->stream, n, omega, delta, x->us[k], x->u[k], x->y[k], x->s[k]);
            if (L > 1) enq_spmv(c, c->A[k], false, x->u[k], x->e[k], epi(1.0, 0.0, nullptr), false);
         }
         if ((rc = ext_fetch_sum(c, &ss))) return rc;
         const double rel = sqrt(ss) / r0_ext;
         if (ext_hist) ext_hist[it] = rel;
         const bool measured = it > 1;            // check_resnorm_flag && loc_iters > 1 (:618)
         omega = 1.0 / (1.0 - omega / mu22);
         it++;
         if (it == num_cycles) break;
         if (measured && rel < tol) break;
      }
   // ---- finish (:777-817) ----
   if ((rc = ext_finish(c, x, r0_ext, ext_relres))) return rc;
   CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
   enq_residual(c);
   if ((rc = amgb_fetch_scalar(c, &ss))) return rc;
   if (relres) *relres = sqrt(ss) / r0;
   float ms = 0;
   CUDA_OK(c, cudaEventSynchronize(c->ev1));
   cudaEventElapsedTime(&ms, c->ev0, c->ev1);
   if (solve_seconds) *solve_seconds = ms * 1e-3;
   if (iters) *iters = it;
   c->r0_norm = r0;
   CUDA_OK(c, cudaGetLastError());
   return AMGB_OK;
}

// ---- asynchronous EXPLICIT extended-system solver (`-solver async_eebpx`) -------------------------------------------------
// SMEM_ExtendedSystemSolve with EXPLICIT_EXTENDED_SYSTEM_BPX and async_flag = 1 (src/SMEM_ExtendedSystem.cpp:295-365 with the
// `#pragma omp barrier`s of :330-332,362-364 skipped; stop rule :636-652): every thread relaxes ITS rows of AA x = bb over and
// over -- r_loc = b - AA x with whatever x the others have written so far, x <- y + omega (delta r ./ diag + x - y), y <- old x,
// its own omega recurrence -- and nobody waits for anybody.  Here a thread is a CTA of a persistent cooperative launch that
// owns a contiguous, nnz-balanced row range (thread.AA_NS / AA_NE); x is shared through L2 (the CTA's L1 is invalidated once
// per sweep by the fence of its leader, so every sweep reads what has reached L2).  Stop: thread 0's sum of the (stale)
// per-thread residual contributions drops below tol * r0_ext (resnorm_converge_flag), or every thread has done num_cycles
// sweeps (threads that are done keep relaxing until the last one is: glob_done_iters == num_threads).
#include "kernels.cuh"

struct ExtAsyncParams {
   DevCSR A;
   const double *b;
   double *x, *y, *r;
   const double *inv_d;            // 1 / a_ii
   const int *row_bounds;          // [grid + 1]
   double delta, mu22, tol2_r0;    // tol^2 * r0_ext^2
   int num_cycles;
   double *cta_r2;                 // [grid] residual contribution of every CTA's last sweep
   volatile int *flag;             // resnorm_converge_flag
   int *done;                      // glob_done_iters
   int *iters;                     // [grid] loc_iters of every CTA at exit
};

namespace {
constexpr int kEBlock = 256;

__global__ void __launch_bounds__(kEBlock) k_async_eebpx(ExtAsyncParams p)
{
   const int cta = blockIdx.x, nct = gridDim.x;
   const int r0 = p.row_bounds[cta], r1 = p.row_bounds[cta + 1];
   DevCSR M = p.A;
   M.rp += r0; M.nrows = r1 - r0;
   SpmvEpilogue e;
   e.alpha = -1.0; e.beta = 1.0; e.gamma = 0.0; e.b = p.b + r0; e.c = nullptr; e.rs = nullptr;
   double omega = 2.0;
   int loc_iters = 1;
   __shared__ int s_stop;
   if (p.num_cycles > 1)
      for (;;) {
         // r_loc = b - AA x on this CTA's rows (vector-per-row CSR; x through L1, refreshed by the fence below)
         csr_rows_dispatch<false, false>(M, p.x, p.r + r0, e, threadIdx.x, kEBlock, false);
         __syncthreads();
         double part = 0.0;
         for (int i = r0 + threadIdx.x; i < r1; i += kEBlock) {
            const double xo = ld_cg(p.x + i), yo = p.y[i], ri = p.r[i];
            st_cg(p.x + i, yo + omega * (p.delta * ri * __ldg(p.inv_d + i) + xo - yo));
            p.y[i] = xo;
            part += ri * ri;
         }
         part = block_sum(part);
         omega = 1.0 / (1.0 - omega / p.mu22);
         loc_iters++;
         if (threadIdx.x == 0) {
            if (loc_iters > 2) *((volatile double *)(p.cta_r2 + cta)) = part;        // check_resnorm_flag && loc_iters > 1 (before the increment)
            __threadfence();                                                         // publishes x; invalidates this SM's L1
            if (cta == 0 && loc_iters > 2) {
               double s = 0.0;
               for (int t = 0; t < nct; t++) s += *((volatile double *)(p.cta_r2 + t));
               if (s < p.tol2_r0) *p.flag = 1;
            }
            int stop = *p.flag;
            if (!stop && loc_iters >= p.num_cycles) {
               if (loc_iters == p.num_cycles) atomicAdd(p.done, 1);
               if (*((volatile int *)p.done) == nct) stop = 1;
            }
            s_stop = stop;
         }
         __syncthreads();
         if (s_stop) break;
      }
   if (threadIdx.x == 0) p.iters[cta] = loc_iters;
}
}  // namespace

// One-level context holding the assembled extended matrix AA (smooth_weight = 1), resident f = bb.  Leaves the extended
// iterate in u (amgb_get_solution); ext_relres = |bb - AA x| / |bb - AA x_0| recomputed after the launch; iters_min / iters_max:
// fewest / most sweeps any CTA performed.
extern "C" int amgb_solve_extended_async(amgb_ctx *c, double tol, int num_cycles, double mu, double delta, int *iters_min, int *iters_max,
                                         double *ext_relres, double *solve_seconds)
{
   NEED_READY(c);
   if (c->L != 1) return amgb_fail(c, AMGB_EINVAL, "the asynchronous extended-system solver runs the EXPLICIT form: a one-level context that holds AA");
   if (num_cycles < 0 || mu == 0.0) return amgb_fail(c, AMGB_EINVAL, "bad arguments");
   const DevCSR &A = c->A[0];
   if (!A.ci || !A.va) return amgb_fail(c, AMGB_EINVAL, "needs the CSR copy of AA (lean_storage = 0)");
   const int n = A.nrows;
   int rc;
   if ((rc = ext_alloc(c))) return rc;
   ExtState *x = c->ext;
   // r0_ext and x_0 = delta r ./ diag (the reference starts from xx = 0: :100-106)
   CUDA_OK(c, cudaMemsetAsync(c->u, 0, sizeof(double) * (size_t)n, c->stream));
   enq_residual(c);
   double ss;
   if ((rc = amgb_fetch_scalar(c, &ss))) return rc;
   const double r0_ext = sqrt(ss);
   c->launches += launch_scale(c->cfg, c->stream, n, c->ws[0], c->r[0], c->u);                        // ws = w / d with w = smooth_weight
   c->launches += launch_axpby(c->cfg, c->stream, n, 0.0, c->r[0], delta / c->opt.smooth_weight, c->u, nullptr);
   CUDA_OK(c, cudaMemsetAsync(x->y[0], 0, sizeof(double) * (size_t)n, c->stream));
   // 1 / a_ii
   c->launches += launch_axpby(c->cfg, c->stream, n, 1.0 / c->opt.smooth_weight, c->ws[0], 0.0, x->us[0], nullptr);
   // CTAs: one cooperative wave, nnz-balanced contiguous row ranges (hypre_LowerBound on the row pointer, src/SMEM_Setup.cpp:870-893)
   int dev = 0, sms = 0, per_sm = 0;
   cudaGetDevice(&dev);
   cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
   cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_async_eebpx, kEBlock, 0);
   int grid = std::max(1, std::min(sms * per_sm, std::max(1, n / 64)));
   std::vector<int> rp((size_t)n + 1);
   CUDA_OK(c, cudaMemcpy(rp.data(), A.rp, sizeof(int) * rp.size(), cudaMemcpyDeviceToHost));
   std::vector<int> bounds((size_t)grid + 1, n);
   bounds[0] = 0;
   const long per = ((long)A.nnz + grid - 1) / grid;
   for (int t = 1; t < grid; t++) bounds[t] = (int)(std::lower_bound(rp.begin(), rp.begin() + n, (int)std::min<long>(per * t, A.nnz)) - rp.begin());
   for (int t = 1; t <= grid; t++) bounds[t] = std::max(bounds[t], bounds[t - 1]);
   int *d_bounds = nullptr, *d_misc = nullptr;
   double *d_r2 = nullptr;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&d_bounds, sizeof(int) * bounds.size(), false))) return rc;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&d_misc, sizeof(int) * ((size_t)grid + 8), true))) return rc;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&d_r2, sizeof(double) * (size_t)grid, false))) return rc;
   CUDA_OK(c, cudaMemcpyAsync(d_bounds, bounds.data(), sizeof(int) * bounds.size(), cudaMemcpyHostToDevice, c->stream));
   std::vector<double> big((size_t)grid, 1e300);          // r_norm2_glob[t] = 100 in the reference (:52): "not measured yet"
   CUDA_OK(c, cudaMemcpyAsync(d_r2, big.data(), sizeof(double) * big.size(), cudaMemcpyHostToDevice, c->stream));
   ExtAsyncParams p;
   p.A = A; p.b = c->f; p.x = c->u; p.y = x->y[0]; p.r = x->r[0]; p.inv_d = x->us[0]; p.row_bounds = d_bounds;
   p.delta = delta; p.mu22 = (2.0 * mu) * (2.0 * mu); p.tol2_r0 = tol * tol * r0_ext * r0_ext; p.num_cycles = num_cycles;
   p.cta_r2 = d_r2; p.flag = d_misc; p.done = d_misc + 1; p.iters = d_misc + 8;
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
   void *args[] = {&p};
   CUDA_OK(c, cudaLaunchCooperativeKernel((void *)k_async_eebpx, dim3(grid), dim3(kEBlock), args, 0, c->stream));
   c->launches += 1;
   CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
   CUDA_OK(c, cudaEventSynchronize(c->ev1));
   float ms = 0;
   cudaEventElapsedTime(&ms, c->ev0, c->ev1);
   if (solve_seconds) *solve_seconds = ms * 1e-3;
   std::vector<int> its((size_t)grid);
   CUDA_OK(c, cudaMemcpy(its.data(), d_misc + 8, sizeof(int) * (size_t)grid, cudaMemcpyDeviceToHost));
   if (iters_min) *iters_min = *std::min_element(its.begin(), its.end());
   if (iters_max) *iters_max = *std::max_element(its.begin(), its.end());
   enq_residual(c);
   if ((rc = amgb_fetch_scalar(c, &ss))) return rc;
   if (ext_relres) *ext_relres = sqrt(ss) / r0_ext;
   CUDA_OK(c, cudaGetLastError());
   return AMGB_OK;
}

// ---- asynchronous IMPLICIT extended-system solver (`-solver async_iebpx`) -------------------------------------------------
// SMEM_ExtendedSystemSolve with IMPLICIT_EXTENDED_SYSTEM_BPX and async_flag = 1 (src/SMEM_Main.cpp:309; the async branches of
// src/SMEM_ExtendedSystem.cpp:305,365,474-479, stop rule :636-652): every level k owns a CTA group of one launch of the
// persistent kernel (k_async_amg<false, true>, async.cu), which plays the reference's thread group of level k.  The group
// loops over its program (async_build_ext_program): it rebuilds the z1 / z2 chains it needs from whatever u_j (j >= k) and
// e_j (j < k) the other groups have written so far, forms r_k, takes its own Chebyshev step on u_k, y_k with its own omega
// recurrence, refreshes e_k, and keeps the count / stop rule -- with no barrier between groups.  Set-up and finish are those of
// amgb_solve_extended.
static int ext_async_prepare(amgb_ctx *c, ExtState *x)
{
   if (x->async_ready) return AMGB_OK;
   const int L = c->L, n0 = c->A[0].nrows;
   const amgb_options &o = c->opt;
   int rc;
   std::vector<AsyncOpSym> sym;
   std::vector<int> op_begin(L + 1, 0);
   for (int q = 0; q < L; q++) {
      op_begin[q] = (int)sym.size();
      if ((rc = async_build_ext_program(o, L, q, sym))) return amgb_fail(c, rc, "no asynchronous extended-system program for these options");
   }
   op_begin[L] = (int)sym.size();
   // CTAs: one cooperative wave, at least one CTA per level group
   const int max_grid = async_max_grid_ext(kABlock);
   if (max_grid < L) return amgb_fail(c, AMGB_EINVAL, "cooperative grid of %d CTAs holds fewer CTAs than the %d level groups", max_grid, L);
   const int grid = std::min(max_grid, std::max(L, n0 / 64 + L));      // small problems: no more CTAs than there is work for
   // ---- the vectors the programs name: the shared per-level vectors are ExtState's; the chains are private to every group
   std::vector<double *> priv((size_t)L * 3 * 64, nullptr);
   auto resolve = [&](int q, int id, double **out) -> int {
      *out = nullptr;
      if (id == AV_NONE) return AMGB_OK;
      const int kind = id / 64, l = id % 64;
      switch (kind) {
         case AV_XF: *out = x->f[l]; return AMGB_OK;
         case AV_XU: *out = x->u[l]; return AMGB_OK;
         case AV_XY: *out = x->y[l]; return AMGB_OK;
         case AV_XE: *out = x->e[l]; return AMGB_OK;
         case AV_WS: *out = c->ws[l]; return AMGB_OK;
         case AV_INVL1: *out = c->inv_l1[l]; return AMGB_OK;
         case AV_XZ1: case AV_XZ2: case AV_XR: break;
         default: return amgb_fail(c, AMGB_EINVAL, "vector kind %d in an extended-system program", kind);
      }
      double *&p = priv[((size_t)q * 3 + (size_t)(kind - AV_XZ1)) * 64 + (size_t)l];
      if (!p) {
         const int r2 = amgb_dev_alloc_bytes(c, (void **)&p, sizeof(double) * (size_t)std::max(1, c->A[l].nrows), true);
         if (r2) return r2;
      }
      *out = p;
      return AMGB_OK;
   };
   std::vector<AsyncOp> dev_ops(sym.size());
   std::vector<double> work(L, 0.0);
   for (int q = 0; q < L; q++)
      for (int i = op_begin[q]; i < op_begin[q + 1]; i++) {
         const AsyncOpSym &s = sym[i];
         AsyncOp &d = dev_ops[i];
         memset(&d, 0, sizeof(d));
         d.type = s.type; d.mat_kind = s.mat_kind; d.mat_level = s.mat_level; d.sval = s.sval; d.range = s.range;
         d.barrier = s.barrier; d.level = s.level; d.sweeps = s.sweeps; d.zero = s.zero; d.locked = s.locked;
         d.e = SpmvEpilogue();
         d.e.alpha = s.alpha; d.e.beta = s.beta; d.e.gamma = s.gamma; d.e.beta2 = s.beta2; d.e.xself = s.xself; d.e.red_scale = s.red_scale;
         double *t;
         if ((rc = resolve(q, s.x, &t))) return rc; d.x = t;
         if ((rc = resolve(q, s.y, &t))) return rc; d.y = t;
         if ((rc = resolve(q, s.b, &t))) return rc; d.e.b = t;
         if ((rc = resolve(q, s.c, &t))) return rc; d.e.c = t;
         if ((rc = resolve(q, s.rs, &t))) return rc; d.e.rs = t;
         if ((rc = resolve(q, s.b2, &t))) return rc; d.e.b2 = t;
         // (xs, red, red_copy, acc: never named by these programs)
         // cost model of the group's program (bytes over the storage's roofline fraction, as for the additive solver):
         // the ratios seed the CTA groups
         if (s.type == AOP_SPMV || s.type == AOP_EXT_RESID) {
            const DevCSR &M = s.mat_kind == AMGB_MAT_A ? c->A[s.mat_level] : (s.mat_kind == AMGB_MAT_P ? c->P[s.mat_level] : c->R[s.mat_level]);
            auto it = c->sell_entries.find(&M);
            work[q] += async_op_cost(M, it == c->sell_entries.end() ? 0 : it->second) + 24.0 * M.nrows;
         } else if (s.type == AOP_EXT_CHEBY) {
            work[q] += 48.0 * c->A[s.level].nrows;
         }
      }
   AsyncParams &hp = x->hp;
   memset(&hp, 0, sizeof(hp));
   hp.num_levels = L;
   hp.first_group = 0;
   hp.smoother = o.smoother;
   hp.n0 = n0;
   for (int l = 0; l < L; l++) {
      hp.A[l] = c->A[l];
      if (l < L - 1) { hp.P[l] = c->P[l]; hp.R[l] = c->R[l]; }
   }
   AsyncOp *d_ops = nullptr;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&d_ops, sizeof(AsyncOp) * dev_ops.size(), false))) return rc;
   CUDA_OK(c, cudaMemcpyAsync(d_ops, dev_ops.data(), sizeof(AsyncOp) * dev_ops.size(), cudaMemcpyHostToDevice, c->stream));
   hp.ops = d_ops;
   for (int q = 0; q <= L; q++) hp.op_begin[q] = op_begin[q];
   async_deal_ctas(work, L, 0, grid, hp.cta_begin);
   hp.slice_ctas = 1;                                   // (no CTA-slice operations in these programs)
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&hp.barrier_count, sizeof(unsigned int) * AMGB_MAX_LEVELS, true))) return rc;
   unsigned int *gen;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&gen, sizeof(unsigned int) * AMGB_MAX_LEVELS, true))) return rc;
   hp.barrier_gen = gen;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&hp.group_stop, sizeof(int) * AMGB_MAX_LEVELS, true))) return rc;
   int *flag;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&flag, sizeof(int) * 4, true))) return rc;
   hp.converge_flag = flag;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&hp.group_ns, sizeof(unsigned long long) * AMGB_MAX_LEVELS, true))) return rc;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&hp.ext.cta_ss, sizeof(double) * (size_t)grid, true))) return rc;
   double *contrib;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&contrib, sizeof(double) * AMGB_MAX_LEVELS, true))) return rc;
   hp.ext.contrib = contrib;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&hp.ext.loc_iters, sizeof(int) * AMGB_MAX_LEVELS, true))) return rc;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&hp.ext.done, sizeof(int) * 4, true))) return rc;
   if ((rc = amgb_dev_alloc_bytes(c, &x->params_dev, sizeof(AsyncParams), false))) return rc;
   if (o.l2_persist && c->arena_used > 0) {
      // the coarse hierarchy pinned in L2 for the launch, as for the additive solver's persistent kernel
      x->window.base_ptr = c->arena;
      x->window.num_bytes = std::min(c->arena_used, c->max_window);
      x->window.hitRatio = 1.0f;
      x->window.hitProp = cudaAccessPropertyPersisting;
      x->window.missProp = cudaAccessPropertyStreaming;
   }
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   x->async_ready = true;
   return AMGB_OK;
}

extern "C" int amgb_solve_extended_implicit_async(amgb_ctx *c, double tol, int num_cycles, double mu, double delta, int *iters,
                                                  double *ext_relres, double *relres, double *group_seconds, double *solve_seconds)
{
   NEED_READY(c);
   const int L = c->L;
   int rc;
   if ((rc = ext_check(c, num_cycles, mu))) return rc;
   if (L > AMGB_MAX_LEVELS) return amgb_fail(c, AMGB_EINVAL, "more than %d levels", AMGB_MAX_LEVELS);
   if ((rc = ext_alloc(c))) return rc;
   ExtState *x = c->ext;
   if ((rc = ext_async_prepare(c, x))) return rc;
   AsyncParams &hp = x->hp;
   double r0, r0_ext, ss;
   if ((rc = ext_setup(c, x, delta, &r0, &r0_ext))) return rc;
   CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
   std::vector<int> it(AMGB_MAX_LEVELS, 1);
   std::vector<unsigned long long> ns(AMGB_MAX_LEVELS, 0);
   if (num_cycles > 1) {                       // (no iteration at all otherwise: every loc_iters stays 1)
      hp.num_cycles = num_cycles;
      hp.ext.delta = delta;
      hp.ext.mu22 = (2.0 * mu) * (2.0 * mu);
      hp.ext.tol = tol;
      hp.ext.r0_ext = r0_ext;
      const std::vector<double> unmeasured(AMGB_MAX_LEVELS, 1e300);     // r_norm2_glob[t] = 100 in the reference (:52)
      CUDA_OK(c, cudaMemcpyAsync((void *)hp.ext.contrib, unmeasured.data(), sizeof(double) * AMGB_MAX_LEVELS, cudaMemcpyHostToDevice, c->stream));
      CUDA_OK(c, cudaMemsetAsync(hp.barrier_count, 0, sizeof(unsigned int) * AMGB_MAX_LEVELS, c->stream));
      CUDA_OK(c, cudaMemsetAsync((void *)hp.barrier_gen, 0, sizeof(unsigned int) * AMGB_MAX_LEVELS, c->stream));
      CUDA_OK(c, cudaMemsetAsync(hp.group_stop, 0, sizeof(int) * AMGB_MAX_LEVELS, c->stream));
      CUDA_OK(c, cudaMemsetAsync((void *)hp.converge_flag, 0, sizeof(int) * 4, c->stream));
      CUDA_OK(c, cudaMemsetAsync(hp.group_ns, 0, sizeof(unsigned long long) * AMGB_MAX_LEVELS, c->stream));
      CUDA_OK(c, cudaMemsetAsync(hp.ext.loc_iters, 0, sizeof(int) * AMGB_MAX_LEVELS, c->stream));
      CUDA_OK(c, cudaMemsetAsync(hp.ext.done, 0, sizeof(int) * 4, c->stream));
      CUDA_OK(c, cudaMemcpyAsync(x->params_dev, &hp, sizeof(AsyncParams), cudaMemcpyHostToDevice, c->stream));
      const int lr = launch_async_ext(c->stream, (const AsyncParams *)x->params_dev, hp.cta_begin[L], kABlock,
                                      x->window.num_bytes > 0 ? &x->window : nullptr);
      if (lr < 0) return amgb_fail(c, AMGB_ECUDA, "cooperative launch failed: %s", cudaGetErrorString((cudaError_t)(-lr)));
      c->launches += 1;
      CUDA_OK(c, cudaMemcpyAsync(it.data(), hp.ext.loc_iters, sizeof(int) * AMGB_MAX_LEVELS, cudaMemcpyDeviceToHost, c->stream));
      CUDA_OK(c, cudaMemcpyAsync(ns.data(), hp.group_ns, sizeof(unsigned long long) * AMGB_MAX_LEVELS, cudaMemcpyDeviceToHost, c->stream));
   }
   // ---- finish (:777-817), as in the synchronous form
   if ((rc = ext_finish(c, x, r0_ext, ext_relres))) return rc;
   CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
   enq_residual(c);
   if ((rc = amgb_fetch_scalar(c, &ss))) return rc;
   if (relres) *relres = sqrt(ss) / r0;
   float ms = 0;
   CUDA_OK(c, cudaEventSynchronize(c->ev1));
   cudaEventElapsedTime(&ms, c->ev0, c->ev1);
   if (solve_seconds) *solve_seconds = ms * 1e-3;
   for (int l = 0; l < L; l++) {
      if (iters) iters[l] = it[l];
      if (group_seconds) group_seconds[l] = 1e-9 * (double)ns[l];
   }
   c->r0_norm = r0;
   CUDA_OK(c, cudaGetLastError());
   return AMGB_OK;
}

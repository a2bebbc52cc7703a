// pcg.cu -- conjugate gradients preconditioned by the selected additive cycle (Multadd / BPX from a zero guess) on one GPU.
// The reference reaches this through hypre's PCG with its cycles as the preconditioner (-hypre_pcg,
// src/DMEM_Setup.cpp:129-167).  The meaning, in this order of operations (tests/pcg_reference.py states the same):
//
//    r = f - A u;  r0 = ||r||;  hist[0] = 1;  r0 == 0 -> no iteration
//    k = 1 .. max_iters:  z = B r;  rho = (r, z)              rho <= 0 or not finite -> breakdown
//                         p = z (k == 1) / z + (rho / rho_old) p;  rho_old = rho
//                         q = A p;  sigma = (p, q)             sigma <= 0 or not finite -> breakdown
//                         u += (rho / sigma) p;  r -= (rho / sigma) q;  hist[k] = ||r|| / r0;  stop when < tol
//    final_relres = ||f - A u|| / r0 (true residual, once)
//
// hypre is not vendored, so parity with hypre_PCGSolve (its stop test and options) is not pinned by reference object code.
//
// Vectors: r = r[0] (enq_cycle reads it and never writes it), z = cvec, p / q allocated on the first call.  One iteration is
// captured once as its own graph (beside the stationary solve's graph_exec):
//   the cycle z = B r with (r, z) fused into its last launch  -> s[PCG_RHO]
//   k_pcg_dir                                                  p = z + beta p
//   q = A_0 p with (p, q) fused                                -> s[PCG_SIGMA]
//   k_pcg_update + reduction                                   u, r, -> s[PCG_RR]
//   one 24-byte D2H of rho, sigma, ||r||^2
// The host tests breakdown and the stop rule after each replay.  On a breakdown k_pcg_update leaves u and r alone.
#include "ctx.h"
#include <cmath>

void amgb_pcg_teardown(amgb_ctx *c)
{
   if (c->pcg_graph) cudaGraphExecDestroy(c->pcg_graph);
   c->pcg_graph = nullptr;
   cudaFree(c->pcg_p);
   cudaFree(c->pcg_q);
   cudaFree(c->pcg_s);
   c->pcg_p = c->pcg_q = c->pcg_s = nullptr;
}

// one iteration, enqueued (captured into the graph)
static void enq_pcg_iteration(amgb_ctx *c)
{
   const int n0 = c->A[0].nrows;
   double *s = c->pcg_s;
   enq_cycle(c, c->cvec, false, c->r[0], s + PCG_RHO);
   c->launches += launch_pcg_dir(c->cfg, c->stream, n0, c->cvec, c->pcg_p, s);
   SpmvEpilogue e;
   e.alpha = 1.0; e.beta = 0.0; e.gamma = 0.0; e.b = nullptr; e.c = nullptr; e.rs = nullptr;
   enq_spmv_dot(c, c->A[0], false, c->pcg_p, c->pcg_q, e, c->pcg_p, s + PCG_SIGMA);
   int grid = 0;
   c->launches += launch_pcg_update(c->cfg, c->stream, n0, c->pcg_p, c->pcg_q, c->u, c->r[0], s, c->partials, &grid);
   c->launches += launch_reduce_partials(c->stream, c->partials, grid, s + PCG_RR);
   cudaMemcpyAsync(c->h_scalars, s, 3 * sizeof(double), cudaMemcpyDeviceToHost, c->stream);
}

extern "C" int amgb_solve_pcg(amgb_ctx *c, double tol, int max_iters, double *hist, int *iters, double *final_relres,
                              double *solve_seconds)
{
   NEED_READY(c);
   const amgb_options &o = c->opt;
   // the preconditioner must be a fixed symmetric linear operator
   if (c->dist) return amgb_fail(c, AMGB_EINVAL, "amgb_solve_pcg runs on a single-GPU context (the row-partitioned form is not implemented)");
   if (o.solver != AMGB_SOLVER_MULTADD && o.solver != AMGB_SOLVER_BPX)
      return amgb_fail(c, AMGB_EINVAL, "amgb_solve_pcg preconditions with the Multadd or BPX cycle (symmetric); this context was set up for solver %d", o.solver);
   if (o.smoother != AMGB_SMOOTH_JACOBI && o.smoother != AMGB_SMOOTH_L1_JACOBI)
      return amgb_fail(c, AMGB_EINVAL, "amgb_solve_pcg needs a symmetric smoother (weighted or L1 Jacobi); smoother %d is not", o.smoother);
   if (o.solver == AMGB_SOLVER_MULTADD && (o.num_pre_smooth_sweeps > 0) != (o.num_post_smooth_sweeps > 0))
      return amgb_fail(c, AMGB_EINVAL, "Multadd with only one of pre / post smoothing has Rbar != Pbar^T: not a symmetric preconditioner");
   if (max_iters < 0) return amgb_fail(c, AMGB_EINVAL, "max_iters < 0");
   const int n0 = c->A[0].nrows;
   int rc;
   if (!c->pcg_p) {
      const size_t bytes = sizeof(double) * ((size_t)n0 + 8);
      CUDA_OK(c, cudaMalloc((void **)&c->pcg_p, bytes));
      CUDA_OK(c, cudaMalloc((void **)&c->pcg_q, bytes));
      CUDA_OK(c, cudaMalloc((void **)&c->pcg_s, sizeof(double) * PCG_NSCALARS));
      c->bytes_allocated += 2 * bytes + sizeof(double) * PCG_NSCALARS;
   }
   // r = f - A u, ||r||^2
   enq_residual(c);
   double ss;
   if ((rc = amgb_fetch_scalar(c, &ss))) return rc;
   const double r0 = sqrt(ss);
   if (hist) hist[0] = 1.0;
   c->r0_norm = r0;
   int done = 0;
   float ms = 0.0f;
   if (r0 > 0.0 && max_iters > 0) {
      if (!c->pcg_graph) {
         cudaGraph_t g;
         const long long before = c->launches;
         CUDA_OK(c, cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
         enq_pcg_iteration(c);
         CUDA_OK(c, cudaStreamEndCapture(c->stream, &g));
         c->pcg_graph_kernels = c->launches - before;
         c->launches = before;
         CUDA_OK(c, cudaGraphInstantiate(&c->pcg_graph, g, 0));
         cudaGraphDestroy(g);
      }
      CUDA_OK(c, cudaMemsetAsync(c->pcg_s, 0, sizeof(double) * PCG_NSCALARS, c->stream));   // PCG_DONE = 0: first direction
      CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
      for (int k = 1; k <= max_iters; k++) {
         CUDA_OK(c, cudaGraphLaunch(c->pcg_graph, c->stream));
         c->launches += c->pcg_graph_kernels;
         CUDA_OK(c, cudaStreamSynchronize(c->stream));
         const double rho = c->h_scalars[0], sigma = c->h_scalars[1], rr = c->h_scalars[2];
         const char *what = nullptr;
         double bad = 0.0;
         if (!(std::isfinite(rho) && rho > 0.0)) { what = "rho = (r, B r)"; bad = rho; }
         else if (!(std::isfinite(sigma) && sigma > 0.0)) { what = "sigma = (p, A p)"; bad = sigma; }
         if (what) {
            if (iters) *iters = done;
            if (final_relres) {
               enq_residual(c);
               if ((rc = amgb_fetch_scalar(c, &ss))) return rc;
               *final_relres = sqrt(ss) / r0;
            }
            if (solve_seconds) *solve_seconds = 0.0;
            return amgb_fail(c, AMGB_ESTATE, "PCG breakdown: %s = %g at iteration %d (B and A must be symmetric positive definite)",
                             what, bad, k);
         }
         done = k;
         const double rel = sqrt(rr) / r0;
         if (hist) hist[k] = rel;
         if (rel < tol) break;
      }
      CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
      CUDA_OK(c, cudaEventSynchronize(c->ev1));
      cudaEventElapsedTime(&ms, c->ev0, c->ev1);
   }
   if (solve_seconds) *solve_seconds = ms * 1e-3;
   if (iters) *iters = done;
   if (final_relres) {
      if (r0 > 0.0) {
         enq_residual(c);
         if ((rc = amgb_fetch_scalar(c, &ss))) return rc;
         *final_relres = sqrt(ss) / r0;
      } else *final_relres = 0.0;
   }
   CUDA_OK(c, cudaGetLastError());
   return AMGB_OK;
}

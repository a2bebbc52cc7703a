// kernels.cu -- stand-alone sm_100a kernels of the additive-AMG solve phase and their launchers.
// Reference loops replaced: SMEM_MatVec / SMEM_SpGEMV / SMEM_Residual (src/SMEM_MatVec.cpp:123-259,
// 302-378), SMEM_Sync_Jacobi / L1Jacobi / SymmetricJacobi / HybridJacobiGaussSeidel
// (src/SMEM_Smooth.cpp:365-443,533-586,643-762), the Chebyshev update and norm of SMEM_Solve
// (src/SMEM_Solve.cpp:179-187,199-203).  All of them are HBM-bound streaming kernels: no tensor
// cores (nothing is a dense contraction).
#include "kernels.cuh"
#include "launch.h"
#include <algorithm>

namespace {

constexpr int kBlock = 256;

// One kernel per storage scheme (separate register budgets): MODE 0 = vector-per-row CSR, 1 = sliced ELL,
// 2 = sliced ELL with the SELL-U encoding (stencil levels); the warp-stream CSR kernel is k_spmv_wstream.
// DOT: the fused per-CTA partial is sum_i y_i * w_i instead of sum_i y_i^2; DUAL: the second output y2 = s2 o (b + y) (kernels.cuh).
// Separate instantiations, so that the others keep their registers.  WIN (MODE 1 on SELL-C-sigma only): the epilogue in row
// order through shared memory (sell_window_rows_cta; spmv_window_path says when).
template <int MODE, bool SVAL, bool DOT = false, bool DUAL = false, bool WIN = false>
__global__ void __launch_bounds__(kBlock, MODE == 2 ? 5 : 1) k_spmv(DevCSR M, const double *x, double *y, SpmvEpilogue e, double *partials,
                                                                    const double *w, double *y2, const double *s2)
{
   const int tid = blockIdx.x * kBlock + threadIdx.x;
   const int tsz = gridDim.x * kBlock;
   const bool norm = partials != nullptr;
   double ss;
   if constexpr (WIN) {
      static_assert(MODE == 1, "the window-staged epilogue is a path of the sliced-ELL kernel");
      __shared__ double sacc[2 * kBlock];
      ss = sell_window_rows_cta<kBlock, SVAL, DOT, DUAL>(M, x, y, e, norm, w, y2, s2, sacc);
   } else if (MODE == 2) ss = sell_rows_team<true, SVAL, 4, true, DOT, DUAL>(M, x, y, e, tid, tsz, norm, w, y2, s2);   // the cached-delta path, 5 CTAs per SM
   else if (MODE == 1) ss = sell_rows_team<true, SVAL, 0, false, DOT, DUAL>(M, x, y, e, tid, tsz, norm, w, y2, s2);
   else ss = csr_rows_dispatch<true, SVAL, DOT, DUAL>(M, x, y, e, tid, tsz, norm, w, y2, s2);
   if (norm) {
      ss = block_sum(ss);
      if (threadIdx.x == 0) partials[blockIdx.x] = ss;
   }
}

__global__ void __launch_bounds__(1024) k_reduce_partials(const double *partials, int n, double *out)
{
   double s = 0.0;
   for (int i = threadIdx.x; i < n; i += blockDim.x) s += partials[i];
   s = block_sum(s);
   if (threadIdx.x == 0) out[0] = s;
}

__global__ void __launch_bounds__(kBlock) k_scale(int n, const double *__restrict__ a, const double *__restrict__ x, double *__restrict__ y)
{
   for (int i = blockIdx.x * kBlock + threadIdx.x; i < n; i += gridDim.x * kBlock) y[i] = a[i] * x[i];
}

__global__ void __launch_bounds__(kBlock) k_add(int n, const double *__restrict__ x, double *__restrict__ y)
{
   for (int i = blockIdx.x * kBlock + threadIdx.x; i < n; i += gridDim.x * kBlock) y[i] += x[i];
}

__global__ void __launch_bounds__(kBlock) k_cheby(int n, double omega, double delta, const double *__restrict__ c,
                                                   double *__restrict__ uo, double *__restrict__ yo, double *__restrict__ u)
{
   for (int i = blockIdx.x * kBlock + threadIdx.x; i < n; i += gridDim.x * kBlock) {
      const double prev = uo[i];
      const double v = yo[i] + omega * (delta * c[i] + prev - yo[i]);
      uo[i] = v;
      yo[i] = prev;
      u[i] = v;
   }
}

__global__ void __launch_bounds__(kBlock) k_sumsq(int n, const double *__restrict__ x, double *partials)
{
   double s = 0.0;
   for (int i = blockIdx.x * kBlock + threadIdx.x; i < n; i += gridDim.x * kBlock) s += x[i] * x[i];
   s = block_sum(s);
   if (threadIdx.x == 0) partials[blockIdx.x] = s;
}

// y = a*x + b*y (b == 0: y is not read); optional copy of the result into z
__global__ void __launch_bounds__(kBlock) k_axpby(int n, double a, const double *x, double b, double *y, double *z)
{
   for (int i = blockIdx.x * kBlock + threadIdx.x; i < n; i += gridDim.x * kBlock) {
      const double v = b == 0.0 ? a * x[i] : a * x[i] + b * y[i];
      y[i] = v;
      if (z) z[i] = v;
   }
}

__global__ void __launch_bounds__(kBlock) k_dot(int n, const double *__restrict__ x, const double *__restrict__ y, double *partials)
{
   double s = 0.0;
   for (int i = blockIdx.x * kBlock + threadIdx.x; i < n; i += gridDim.x * kBlock) s += x[i] * y[i];
   s = block_sum(s);
   if (threadIdx.x == 0) partials[blockIdx.x] = s;
}

// preconditioned conjugate gradients (csrc/pcg.cu): every CTA reads the scalars the previous reductions left in s[PCG_*]
// (no host round trip).  p = z + beta p, beta = rho / rho_old, and p = z outright on the first iteration (0 * p would keep a
// NaN an earlier solve left in p).
__global__ void __launch_bounds__(kBlock) k_pcg_dir(int n, const double *__restrict__ z, double *__restrict__ p, const double *s)
{
   const bool first = s[PCG_DONE] == 0.0;
   const double beta = first ? 0.0 : s[PCG_RHO] / s[PCG_RHO_OLD];
   for (int i = blockIdx.x * kBlock + threadIdx.x; i < n; i += gridDim.x * kBlock) p[i] = first ? z[i] : z[i] + beta * p[i];
}

// alpha = rho / sigma; u += alpha p; r -= alpha q; partial sums of r_i^2.  On a breakdown (rho or sigma not positive and
// finite) u and r are left as they are, so that they hold the completed iterations.  CTA 0 then records rho as rho_old and
// counts the iteration (the other CTAs never read those two slots in this launch).
__global__ void __launch_bounds__(kBlock) k_pcg_update(int n, const double *__restrict__ p, const double *__restrict__ q,
                                                       double *__restrict__ u, double *__restrict__ r, double *s, double *partials)
{
   const double rho = s[PCG_RHO], sigma = s[PCG_SIGMA];
   const bool ok = isfinite(rho) && rho > 0.0 && isfinite(sigma) && sigma > 0.0;
   const double alpha = rho / sigma;
   double ss = 0.0;
   for (int i = blockIdx.x * kBlock + threadIdx.x; i < n; i += gridDim.x * kBlock) {
      double ri = r[i];
      if (ok) {
         u[i] += alpha * p[i];
         ri -= alpha * q[i];
         r[i] = ri;
      }
      ss += ri * ri;
   }
   ss = block_sum(ss);
   if (threadIdx.x == 0) {
      partials[blockIdx.x] = ss;
      if (blockIdx.x == 0 && ok) {
         s[PCG_RHO_OLD] = rho;
         s[PCG_DONE] += 1.0;
      }
   }
}

// u += e on this GPU and on every peer GPU (their u mapped through CUDA IPC): the `#pragma omp atomic` of
// src/SMEM_Async_AMG.cpp:297 / the accumulate-on-receive of src/DMEM_Comm.cpp:267-330 as fire-and-forget
// red.global.add.f64 over NVLink -- no message queues, no in-flight accounting, nobody waits for anybody
__global__ void __launch_bounds__(kBlock) k_push_correction(int n, const double *__restrict__ e, double *u, PeerPtrs peers)
{
   for (int i = blockIdx.x * kBlock + threadIdx.x; i < n; i += gridDim.x * kBlock) {
      const double v = e[i];
      red_add_f64(u + i, v);
      for (int p = 0; p < peers.n; p++) red_add_f64(peers.p[p] + i, v);
   }
}

// hybrid Jacobi / Gauss-Seidel over an EXPLICIT block list (amgb_set_jgs_blocks): block b = rows [bounds[b], bounds[b+1]), one thread
// walks one block in row order -- the arithmetic of hybrid_jgs_team (src/SMEM_Smooth.cpp:533-586) with the reference's own blocks
// (a thread's nnz-balanced row range, src/SMEM_Setup.cpp:954-959).  A parity path: with the reference's few, huge blocks it is
// as sequential as the reference's threads are.
__global__ void __launch_bounds__(kBlock) k_hybrid_jgs_list(DevCSR A, const double *f, double *u, const double *u_prev,
                                                            const double *scale, const int *__restrict__ bounds, int nblocks, int zero_guess)
{
   for (int blk = blockIdx.x * kBlock + threadIdx.x; blk < nblocks; blk += gridDim.x * kBlock) {
      const int ns = bounds[blk], ne = bounds[blk + 1];
      if (zero_guess)
         for (int i = ns; i < ne; i++) u[i] = 0.0;
      for (int i = ns; i < ne; i++) {
         const int s = A.rp[i], t = A.rp[i + 1];
         const double d = A.va[s];
         if (d != 0.0) {
            double res = f[i];
            for (int p = s; p < t; p++) {
               const int ii = A.ci[p];
               if (ii >= ns && ii < ne) res -= A.va[p] * u[ii];
               else if (!zero_guess) res -= A.va[p] * u_prev[ii];
            }
            const double div = scale ? scale[i] : d;
            if (zero_guess) u[i] = res / div;
            else u[i] += res / div;
         }
      }
   }
}

__global__ void __launch_bounds__(kBlock) k_hybrid_jgs(DevCSR A, const double *f, double *u, const double *u_prev,
                                                        const double *scale, int B, int zero_guess)
{
   hybrid_jgs_team<true>(A, f, u, u_prev, scale, B, zero_guess != 0, blockIdx.x * kBlock + threadIdx.x, gridDim.x * kBlock);
}

template <int LPB>
__global__ void __launch_bounds__(kBlock) k_hybrid_jgs_sw(DevCSR A, const double *f, double *u, const double *u_prev,
                                                           const double *scale, int B, int zero_guess)
{
   __shared__ double ub[(kBlock / LPB) * AMGB_JGS_BMAX];
   hybrid_jgs_subwarp_team<true, LPB>(A, f, u, u_prev, scale, B, zero_guess != 0, blockIdx.x * kBlock + threadIdx.x,
                                      gridDim.x * kBlock, ub);
}

__global__ void __launch_bounds__(kBlock) k_async_gs(DevCSR A, const double *f, double *u, int B, int sweeps)
{
   async_gs_team<true>(A, f, u, B, sweeps, blockIdx.x * kBlock + threadIdx.x, gridDim.x * kBlock);
}

__global__ void __launch_bounds__(kBlock) k_spmv_transpose(DevCSR M, const double *x, double *y)
{
   csr_transpose_rows_team<8>(M, x, y, blockIdx.x * kBlock + threadIdx.x, gridDim.x * kBlock);
}

__global__ void __launch_bounds__(kBlock) k_diag_scale(DevCSR A, double w, double *ws, double *dow)
{
   for (int i = blockIdx.x * kBlock + threadIdx.x; i < A.nrows; i += gridDim.x * kBlock) {
      const double d = (A.rp[i + 1] > A.rp[i]) ? A.va[A.rp[i]] : 0.0;
      ws[i] = (d != 0.0) ? w / d : 0.0;
      if (dow) dow[i] = d / w;
   }
}

// lean storage: the same scale arrays from the diagonal / l1 norms the host formed at upload
__global__ void __launch_bounds__(kBlock) k_diag_scale_vec(int n, const double *__restrict__ diag, const double *__restrict__ l1src, double w,
                                                            double *ws, double *dow, double *l1, double *inv_l1)
{
   for (int i = blockIdx.x * kBlock + threadIdx.x; i < n; i += gridDim.x * kBlock) {
      const double d = diag[i], s = l1src[i];
      ws[i] = (d != 0.0) ? w / d : 0.0;
      dow[i] = d / w;
      l1[i] = s;
      inv_l1[i] = (s != 0.0) ? 1.0 / s : 0.0;
   }
}

__global__ void __launch_bounds__(kBlock) k_l1(DevCSR A, double *l1, double *inv_l1)
{
   for (int i = blockIdx.x * kBlock + threadIdx.x; i < A.nrows; i += gridDim.x * kBlock) {
      double s = 0.0;
      for (int p = A.rp[i]; p < A.rp[i + 1]; p++) s += fabs(A.va[p]);
      l1[i] = s;
      inv_l1[i] = (s != 0.0) ? 1.0 / s : 0.0;
   }
}

__global__ void __launch_bounds__(kBlock) k_colscale(int nnz, const int *__restrict__ ci, const double *__restrict__ va,
                                                      const double *__restrict__ cs, double *__restrict__ out)
{
   for (int p = blockIdx.x * kBlock + threadIdx.x; p < nnz; p += gridDim.x * kBlock) out[p] = va[p] * cs[ci[p]];
}

inline int grid_for(const LaunchCfg &cfg, long work_threads)
{
   long g = (work_threads + kBlock - 1) / kBlock;
   long cap = (long)cfg.num_sms * cfg.ctas_per_sm;
   return (int)std::max(1L, std::min(g, cap));
}

}  // namespace

template <bool SVAL, bool DOT = false, bool DUAL = false>
__global__ void __launch_bounds__(kBlock) k_spmv_wstream(DevCSR M, const double *x, double *y, SpmvEpilogue e, double *partials, const double *w,
                                                         double *y2, const double *s2)
{
   __shared__ __align__(16) double swarp[(kBlock / 32) * AMGB_WARP_CHUNK];
   const bool norm = partials != nullptr;
   const int warp = threadIdx.x >> 5;
   double ss = warp_stream_rows_team<true, SVAL, DOT, DUAL>(M, x, y, e, blockIdx.x * (kBlock / 32) + warp, gridDim.x * (kBlock / 32),
                                                            swarp + warp * AMGB_WARP_CHUNK, norm, w, y2, s2);
   if (norm) {
      ss = block_sum(ss);
      if (threadIdx.x == 0) partials[blockIdx.x] = ss;
   }
}

template <class K>
static int resident_ctas(K kernel, int block, int num_sms, int *cache)
{
   // co-resident CTAs of this kernel on the device: grids are sized to exactly one wave
   if (*cache == 0) {
      int v = 0;
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, kernel, block, 0) != cudaSuccess || v < 1) v = 1;
      *cache = std::min(v, 8);      // the per-CTA partial sums of the fused norms are sized for 8 CTAs per SM (LaunchCfg::ctas_per_sm)
   }
   return num_sms * *cache;
}

// (per instantiation: a function template has one set of statics per instantiation)
template <int MODE, bool SVAL, bool DOT, bool DUAL = false, bool WIN = false>
static int spmv_mode_go(const LaunchCfg &cfg, cudaStream_t st, const DevCSR &M, const double *x, double *y, const SpmvEpilogue &e,
                        double *partials, long ctas_of_work, const double *w, double *y2 = nullptr, const double *s2 = nullptr)
{
   static int occ = 0;
   const int cap = resident_ctas(k_spmv<MODE, SVAL, DOT, DUAL, WIN>, kBlock, cfg.num_sms, &occ);
   const int grid = (int)std::max(1L, std::min(ctas_of_work, (long)cap));
   k_spmv<MODE, SVAL, DOT, DUAL, WIN><<<grid, kBlock, 0, st>>>(M, x, y, e, partials, w, y2, s2);
   return grid;
}
template <int MODE, bool WIN = false>
static int launch_spmv_mode(const LaunchCfg &cfg, cudaStream_t st, const DevCSR &M, bool use_sval, const double *x, double *y,
                            const SpmvEpilogue &e, double *partials, long ctas_of_work, const double *w, double *y2, const double *s2)
{
   if (y2) return spmv_mode_go<MODE, true, false, true, WIN>(cfg, st, M, x, y, e, nullptr, ctas_of_work, nullptr, y2, s2);
   if (w) return use_sval ? spmv_mode_go<MODE, true, true, false, WIN>(cfg, st, M, x, y, e, partials, ctas_of_work, w)
                          : spmv_mode_go<MODE, false, true, false, WIN>(cfg, st, M, x, y, e, partials, ctas_of_work, w);
   return use_sval ? spmv_mode_go<MODE, true, false, false, WIN>(cfg, st, M, x, y, e, partials, ctas_of_work, nullptr)
                   : spmv_mode_go<MODE, false, false, false, WIN>(cfg, st, M, x, y, e, partials, ctas_of_work, nullptr);
}

// The window-staged epilogue (sell_window_rows_cta) needs a SELL-C-sigma matrix whose sorting windows never straddle the
// kBlock slots a CTA takes per iteration: sigma divides kBlock and the view starts at a multiple of kBlock / 32 slices.
bool spmv_window_path(const LaunchCfg &cfg, const DevCSR &M)
{
   return M.sell_perm && !M.su_desc && M.sell_slices > 0 && cfg.sell_window_sigma > 1 && kBlock % cfg.sell_window_sigma == 0 &&
          M.sell_base % (kBlock / 32) == 0;
}

template <bool SVAL, bool DOT, bool DUAL = false>
static int wstream_go(const LaunchCfg &cfg, cudaStream_t st, const DevCSR &M, const double *x, double *y, const SpmvEpilogue &e,
                      double *partials, const double *w, double *y2 = nullptr, const double *s2 = nullptr)
{
   static int occ = 0;
   const int cap = resident_ctas(k_spmv_wstream<SVAL, DOT, DUAL>, kBlock, cfg.num_sms, &occ);
   const long want = ((long)M.nblk + kBlock / 32 - 1) / (kBlock / 32);
   const int grid = (int)std::max(1L, std::min(want, (long)cap));
   k_spmv_wstream<SVAL, DOT, DUAL><<<grid, kBlock, 0, st>>>(M, x, y, e, partials, w, y2, s2);
   return grid;
}
static int launch_wstream(const LaunchCfg &cfg, cudaStream_t st, const DevCSR &M, bool use_sval, const double *x, double *y,
                          const SpmvEpilogue &e, double *partials, const double *w, double *y2, const double *s2)
{
   if (y2) return wstream_go<true, false, true>(cfg, st, M, x, y, e, nullptr, nullptr, y2, s2);
   if (w) return use_sval ? wstream_go<true, true>(cfg, st, M, x, y, e, partials, w)
                          : wstream_go<false, true>(cfg, st, M, x, y, e, partials, w);
   return use_sval ? wstream_go<true, false>(cfg, st, M, x, y, e, partials, nullptr)
                   : wstream_go<false, false>(cfg, st, M, x, y, e, partials, nullptr);
}

int launch_spmv(const LaunchCfg &cfg, cudaStream_t st, const DevCSR &M, bool use_sval, const double *x, double *y,
                const SpmvEpilogue &e, double *partials, int *grid_out, const double *dot_w, double *y2, const double *s2)
{
   int grid;
   if (M.sell_slices > 0 && M.su_desc) grid = launch_spmv_mode<2>(cfg, st, M, use_sval, x, y, e, partials, ((long)M.sell_slices * 32 + kBlock - 1) / kBlock, dot_w, y2, s2);
   else if (spmv_window_path(cfg, M))
      grid = launch_spmv_mode<1, true>(cfg, st, M, use_sval, x, y, e, partials, ((long)M.sell_slices * 32 + kBlock - 1) / kBlock, dot_w, y2, s2);
   else if (M.sell_slices > 0) grid = launch_spmv_mode<1>(cfg, st, M, use_sval, x, y, e, partials, ((long)M.sell_slices * 32 + kBlock - 1) / kBlock, dot_w, y2, s2);
   else if (M.nblk > 0) grid = launch_wstream(cfg, st, M, use_sval, x, y, e, partials, dot_w, y2, s2);
   else grid = launch_spmv_mode<0>(cfg, st, M, use_sval, x, y, e, partials, ((long)M.nrows * M.lpr + kBlock - 1) / kBlock, dot_w, y2, s2);
   if (grid_out) *grid_out = grid;
   return 1;
}

int spmv_units(const DevCSR &M) { return M.sell_slices > 0 ? M.sell_slices : (M.nblk > 0 ? M.nblk : M.nrows); }

// the same product restricted to launch units [u0, u1) (slices / chunks / rows, whichever the storage uses)
int launch_spmv_units(const LaunchCfg &cfg, cudaStream_t st, const DevCSR &M, int u0, int u1, bool use_sval, const double *x,
                      double *y, const SpmvEpilogue &e, double *partials, int *grid_out, const double *dot_w)
{
   if (grid_out) *grid_out = 0;
   if (u1 <= u0) return 0;
   // a view that ends inside a CTA's slots would have the window-staged epilogue write rows of slots outside the view
   LaunchCfg cv = cfg;
   cv.sell_window_sigma = 0;
   DevCSR V = M;
   SpmvEpilogue ev = e;
   double *yv = y;
   if (M.sell_slices > 0) { V.sell_off += u0; V.sell_base += u0; V.sell_slices = u1 - u0; if (V.su_desc) V.su_desc += u0; }
   else if (M.nblk > 0) { V.blk += u0; V.nblk = u1 - u0; }
   else {
      V.rp += u0; V.nrows = u1 - u0; yv += u0;
      if (ev.b) ev.b += u0;
      if (ev.c) ev.c += u0;
      if (ev.rs) ev.rs += u0;
      if (ev.b2) ev.b2 += u0;
      if (ev.xs) ev.xs += u0;
      if (dot_w) dot_w += u0;
   }
   return launch_spmv(cv, st, V, use_sval, x, yv, ev, partials, grid_out, dot_w);
}

int launch_reduce_partials(cudaStream_t st, const double *partials, int n, double *out)
{
   k_reduce_partials<<<1, 1024, 0, st>>>(partials, n, out);
   return 1;
}

int launch_scale(const LaunchCfg &cfg, cudaStream_t st, int n, const double *a, const double *x, double *y)
{
   k_scale<<<grid_for(cfg, n), kBlock, 0, st>>>(n, a, x, y);
   return 1;
}

int launch_add(const LaunchCfg &cfg, cudaStream_t st, int n, const double *x, double *y)
{
   k_add<<<grid_for(cfg, n), kBlock, 0, st>>>(n, x, y);
   return 1;
}

int launch_cheby(const LaunchCfg &cfg, cudaStream_t st, int n, double omega, double delta, const double *c,
                 double *u_outer, double *y_outer, double *u)
{
   k_cheby<<<grid_for(cfg, n), kBlock, 0, st>>>(n, omega, delta, c, u_outer, y_outer, u);
   return 1;
}

int launch_axpby(const LaunchCfg &cfg, cudaStream_t st, int n, double a, const double *x, double b, double *y, double *z)
{
   k_axpby<<<grid_for(cfg, n), kBlock, 0, st>>>(n, a, x, b, y, z);
   return 1;
}

int launch_dot(const LaunchCfg &cfg, cudaStream_t st, int n, const double *x, const double *y, double *partials, int *grid_out)
{
   int grid = grid_for(cfg, n);
   if (grid_out) *grid_out = grid;
   k_dot<<<grid, kBlock, 0, st>>>(n, x, y, partials);
   return 1;
}

int launch_pcg_dir(const LaunchCfg &cfg, cudaStream_t st, int n, const double *z, double *p, const double *s)
{
   k_pcg_dir<<<grid_for(cfg, n), kBlock, 0, st>>>(n, z, p, s);
   return 1;
}

int launch_pcg_update(const LaunchCfg &cfg, cudaStream_t st, int n, const double *p, const double *q, double *u, double *r,
                      double *s, double *partials, int *grid_out)
{
   const int grid = grid_for(cfg, n);
   if (grid_out) *grid_out = grid;
   k_pcg_update<<<grid, kBlock, 0, st>>>(n, p, q, u, r, s, partials);
   return 1;
}

int launch_push_correction(const LaunchCfg &cfg, cudaStream_t st, int n, const double *e, double *u, const PeerPtrs &peers)
{
   k_push_correction<<<grid_for(cfg, n), kBlock, 0, st>>>(n, e, u, peers);
   return 1;
}

int launch_sumsq(const LaunchCfg &cfg, cudaStream_t st, int n, const double *x, double *partials, int *grid_out)
{
   int grid = grid_for(cfg, n);
   if (grid_out) *grid_out = grid;
   k_sumsq<<<grid, kBlock, 0, st>>>(n, x, partials);
   return 1;
}

int launch_hybrid_jgs(const LaunchCfg &cfg, cudaStream_t st, const DevCSR &A, const double *f, double *u,
                      const double *u_prev, const double *scale, int block_rows, bool zero_guess)
{
   long nblocks = ((long)A.nrows + block_rows - 1) / block_rows;
   if (block_rows <= AMGB_JGS_BMAX && A.nrows > 0) {
      // lanes per block from the mean row length; one sub-warp per block
      const double avg = (double)A.nnz / A.nrows;
      const int z = zero_guess ? 1 : 0;
      if (avg <= 5.0) k_hybrid_jgs_sw<4><<<grid_for(cfg, nblocks * 4), kBlock, 0, st>>>(A, f, u, u_prev, scale, block_rows, z);
      else if (avg <= 10.0) k_hybrid_jgs_sw<8><<<grid_for(cfg, nblocks * 8), kBlock, 0, st>>>(A, f, u, u_prev, scale, block_rows, z);
      else if (avg <= 20.0) k_hybrid_jgs_sw<16><<<grid_for(cfg, nblocks * 16), kBlock, 0, st>>>(A, f, u, u_prev, scale, block_rows, z);
      else k_hybrid_jgs_sw<32><<<grid_for(cfg, nblocks * 32), kBlock, 0, st>>>(A, f, u, u_prev, scale, block_rows, z);
      return 1;
   }
   k_hybrid_jgs<<<grid_for(cfg, nblocks), kBlock, 0, st>>>(A, f, u, u_prev, scale, block_rows, zero_guess ? 1 : 0);
   return 1;
}

int launch_hybrid_jgs_list(const LaunchCfg &cfg, cudaStream_t st, const DevCSR &A, const double *f, double *u,
                           const double *u_prev, const double *scale, const int *bounds, int nblocks, bool zero_guess)
{
   k_hybrid_jgs_list<<<grid_for(cfg, nblocks), kBlock, 0, st>>>(A, f, u, u_prev, scale, bounds, nblocks, zero_guess ? 1 : 0);
   return 1;
}

int launch_async_gs(const LaunchCfg &cfg, cudaStream_t st, const DevCSR &A, const double *f, double *u, int block_rows,
                    int sweeps, bool semi)
{
   const long nblocks = ((long)A.nrows + block_rows - 1) / block_rows;
   const int grid = grid_for(cfg, nblocks);
   if (!semi) { k_async_gs<<<grid, kBlock, 0, st>>>(A, f, u, block_rows, sweeps); return 1; }
   for (int k = 0; k < sweeps; k++) k_async_gs<<<grid, kBlock, 0, st>>>(A, f, u, block_rows, 1);
   return sweeps;
}

int launch_spmv_transpose(const LaunchCfg &cfg, cudaStream_t st, const DevCSR &M, const double *x, double *y)
{
   cudaMemsetAsync(y, 0, sizeof(double) * (size_t)M.ncols, st);
   k_spmv_transpose<<<grid_for(cfg, (long)M.nrows * 8), kBlock, 0, st>>>(M, x, y);
   return 1;
}

int launch_diag_scale(cudaStream_t st, const DevCSR &A, double w, double *ws, double *dow)
{
   LaunchCfg cfg;
   k_diag_scale<<<grid_for(cfg, A.nrows), kBlock, 0, st>>>(A, w, ws, dow);
   return 1;
}

int launch_diag_scale_vec(cudaStream_t st, int n, const double *diag, const double *l1src, double w, double *ws, double *dow,
                          double *l1, double *inv_l1)
{
   LaunchCfg cfg;
   k_diag_scale_vec<<<grid_for(cfg, n), kBlock, 0, st>>>(n, diag, l1src, w, ws, dow, l1, inv_l1);
   return 1;
}

int launch_l1(cudaStream_t st, const DevCSR &A, double *l1, double *inv_l1)
{
   LaunchCfg cfg;
   k_l1<<<grid_for(cfg, A.nrows), kBlock, 0, st>>>(A, l1, inv_l1);
   return 1;
}

int launch_colscale(cudaStream_t st, int nnz, const int *ci, const double *va, const double *cs, double *out)
{
   LaunchCfg cfg;
   k_colscale<<<grid_for(cfg, nnz), kBlock, 0, st>>>(nnz, ci, va, cs, out);
   return 1;
}

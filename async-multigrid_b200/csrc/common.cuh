// common.cuh -- shared device helpers for the sm_100a additive-AMG kernels.
#pragma once
#include <cuda_runtime.h>

#define AMGB_WARP 32
#define AMGB_FULL 0xffffffffu

// Device-resident CSR matrix (row_ptr/col/val in HBM).  `sval` is an optional second value
// array with the same pattern: A*diag(w/d) (or A*diag(1/l1)), which turns the reference's
// three-pass symmetrised Jacobi (src/SMEM_Smooth.cpp:643-702) into ONE SpMV-shaped pass.
// `sell_*`: optional sliced-ELL (C = 32) copy used by the stencil-level kernels.
struct DevCSR {
   int nrows = 0, ncols = 0, nnz = 0;
   const int *rp = nullptr;
   const int *ci = nullptr;
   const double *va = nullptr;
   const double *sval = nullptr;
   // sliced ELL, slice height 32: slice s holds rows [32s, 32s+32); entry k of row r sits at
   // sell_off[s] + k*32 + (r & 31); padded entries have col = row's own index and val = 0.
   int sell_slices = 0;
   const int *sell_off = nullptr;    // [slices+1] offsets in units of entries
   const int *sell_ci = nullptr;
   const double *sell_va = nullptr;
   const double *sell_sval = nullptr;
   int sell_base = 0;                // index of the first slice of this view (row-range launches of the multi-GPU path)
   const int *sell_perm = nullptr;   // SELL-C-sigma: slot (32*slice + lane) -> row, -1 for padding slots; nullptr = identity
   // SELL-U ("uniform slices", sigma = 1 only): a lossless second encoding of a slice whose entries take few distinct
   // (column - row, value) pairs -- the stencil levels, where every row of a slice carries the same 7 / 27 pairs.  Slice s
   // owns groups [su_desc[s].x, su_desc[s].x + su_desc[s].y) of a DEDUPLICATED group table (slices with the same list share
   // it: a stencil has a few dozen distinct lists, which then live in L1); group g = {delta, lane mask} + value (+ the
   // column-scaled value): lane l adds value * x[row + delta] when bit l of the mask is set.  The kernel streams the vectors
   // only.  su_desc[s].y == 0: the slice is not encoded, the regular arrays are used.
   const int2 *su_desc = nullptr;    // [slices] {first group, number of groups}
   const int2 *su_dm = nullptr;      // {column - row, lane mask}
   const double *su_va = nullptr;
   const double *su_sval = nullptr;
   int lpr = 8;                      // lanes per row chosen for the CSR vector kernel
   // warp-stream row chunks (warp_stream_rows_team): consecutive rows whose entries fit AMGB_WARP_CHUNK; a row longer
   // than that is a chunk of its own, reduced by the whole warp.  Also the launch units of the multi-GPU interior split.
   int nblk = 0;
   const int4 *blk = nullptr;        // per chunk {first row, end row, first entry, end entry}
   // multi-GPU: launch units (slices / chunks / rows) [ulo, uhi) read only OWNED entries of the input vector, so
   // they can run while the halo exchange is in flight; the units outside wait for it.  uhi <= ulo: no split.
   int ulo = 0, uhi = 0;
};
#define AMGB_WARP_CHUNK 256           // largest warp-stream chunk, in entries (8 per lane)

// y_i = gamma*c_i + rs_i * (beta*b_i + alpha * sum_j M_ij x_j)       (rs == nullptr -> 1)
// covers: MatVec (alpha=1), Residual (alpha=-1,beta=1,b=f), prolong-and-add (beta=1,b=y),
// general Jacobi sweep (rs=w/d, alpha=-1, beta=1, b=f, gamma=1, c=u_prev),
// symmetrised Jacobi from zero guess with M = A*diag(w/d) (rs=w/d, alpha=-1, beta=2, b=r).
// optional extras (level-0 factorised transfers): a second vector inside the scaled bracket and the input's own
// entry outside it:  y_i = gamma*c_i + rs_i*(beta*b_i + beta2*b2_i + alpha*sum_j M_ij x_j) + xself*xs_i
struct SpmvEpilogue {
   double alpha, beta, gamma;
   const double *b;
   const double *c;
   const double *rs;
   double beta2 = 0.0, xself = 0.0;
   const double *b2 = nullptr;
   const double *xs = nullptr;
   // persistent asynchronous kernel only (RO == false): the row result is also (or only, y == nullptr) reduced into a vector
   // that other CTA groups update concurrently, red_i += red_scale * y_i with red.global.add.f64 (the `omp atomic` of
   // src/SMEM_Async_AMG.cpp:297), the group's private copy red_copy_i = red_i is taken right after (:298), and acc_i += y_i
   // keeps the group's accumulated correction (-read_type res, :288)
   double red_scale = 1.0;
   double *red = nullptr;
   double *red_copy = nullptr;
   double *acc = nullptr;
};

__device__ __forceinline__ double ld_stream(const double *p)
{
   // matrix values / indices are read exactly once: keep them out of L1
   double v;
   asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
   return v;
}
__device__ __forceinline__ int ld_stream(const int *p)
{
   int v;
   asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
   return v;
}
// coherent (L2) load for vectors that other CTA groups update concurrently inside the persistent
// asynchronous kernel
__device__ __forceinline__ double ld_cg(const double *p)
{
   double v;
   asm volatile("ld.global.cg.f64 %0, [%1];" : "=d"(v) : "l"(p));
   return v;
}
// L1-cached load on the coherent path (NOT ld.global.nc): see ld_x<false> in kernels.cuh.  Inline PTX so that a
// `const __restrict__` qualifier cannot turn it into a non-coherent load behind our back.
__device__ __forceinline__ double ld_ca(const double *p)
{
   double v;
   asm volatile("ld.global.ca.f64 %0, [%1];" : "=d"(v) : "l"(p));
   return v;
}
__device__ __forceinline__ void st_cg(double *p, double v)
{
   asm volatile("st.global.cg.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}
// fire-and-forget fp64 reduction into global memory (#pragma omp atomic, src/SMEM_Async_AMG.cpp:297)
__device__ __forceinline__ void red_add_f64(double *p, double v)
{
   asm volatile("red.global.add.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}

template <int W>
__device__ __forceinline__ double subwarp_sum(double v)
{
#pragma unroll
   for (int o = W / 2; o > 0; o >>= 1) v += __shfl_down_sync(AMGB_FULL, v, o, W);
   return v;
}

// RO: operands are read-only for the whole launch (stand-alone kernels); otherwise they may have
// been written by other CTAs earlier in the same persistent launch and are read from L2.
template <bool RO>
__device__ __forceinline__ double epilogue_apply(const SpmvEpilogue &e, int row, double ax)
{
   double t = e.alpha * ax;
   if (e.b) t += e.beta * (RO ? e.b[row] : ld_cg(e.b + row));
   if (e.b2) t += e.beta2 * (RO ? e.b2[row] : ld_cg(e.b2 + row));
   if (e.rs) t *= __ldg(e.rs + row);
   if (e.c) t += e.gamma * (RO ? e.c[row] : ld_cg(e.c + row));
   if (e.xs) t += e.xself * (RO ? e.xs[row] : ld_cg(e.xs + row));
   return t;
}

// store of a finished row: plain store for the stand-alone kernels; inside the persistent kernel optionally the fused
// "u += e; u_k = u" of the asynchronous update
template <bool RO>
__device__ __forceinline__ void epilogue_store(const SpmvEpilogue &e, double *y, int row, double v)
{
   if (!RO) {
      if (e.red) {
         red_add_f64(e.red + row, e.red_scale * v);
         if (e.red_copy) e.red_copy[row] = ld_cg(e.red + row);
      }
      if (e.acc) e.acc[row] += v;
      if (y) y[row] = v;
   } else {
      y[row] = v;
   }
}

// epilogue with the row operands loaded ahead of the reduction (latency off the critical path)
struct EpiOps { double b, c, rs, b2 = 0.0, xs = 0.0; };
template <bool RO>
__device__ __forceinline__ EpiOps epilogue_load(const SpmvEpilogue &e, int row)
{
   EpiOps o;
   o.b = e.b ? (RO ? e.b[row] : ld_cg(e.b + row)) : 0.0;
   o.rs = e.rs ? __ldg(e.rs + row) : 1.0;
   o.c = e.c ? (RO ? e.c[row] : ld_cg(e.c + row)) : 0.0;
   o.b2 = e.b2 ? (RO ? e.b2[row] : ld_cg(e.b2 + row)) : 0.0;
   o.xs = e.xs ? (RO ? e.xs[row] : ld_cg(e.xs + row)) : 0.0;
   return o;
}
__device__ __forceinline__ double epilogue_finish(const SpmvEpilogue &e, const EpiOps &o, double ax)
{
   double t = e.alpha * ax;
   if (e.b) t += e.beta * o.b;
   if (e.b2) t += e.beta2 * o.b2;
   if (e.rs) t *= o.rs;
   if (e.c) t += e.gamma * o.c;
   if (e.xs) t += e.xself * o.xs;
   return t;
}

// block-wide sum; result valid in thread 0.  blockDim.x multiple of 32, <= 1024.
__device__ __forceinline__ double block_sum(double v)
{
   __shared__ double sm[32];
   v = subwarp_sum<32>(v);
   int w = threadIdx.x >> 5, l = threadIdx.x & 31;
   if (l == 0) sm[w] = v;
   __syncthreads();
   if (w == 0) {
      v = (l < (blockDim.x >> 5)) ? sm[l] : 0.0;
      v = subwarp_sum<32>(v);
   }
   __syncthreads();
   return v;
}

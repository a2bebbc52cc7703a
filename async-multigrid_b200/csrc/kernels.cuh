// kernels.cuh -- device-side building blocks shared by the stand-alone kernels (kernels.cu) and
// the persistent asynchronous kernel (async.cu).  A "team" is the set of threads that cooperates
// on one operation: the whole grid for a stand-alone launch, one level's CTA group inside the
// persistent kernel (the reference's thread group of a level, src/SMEM_Setup.cpp:855-868).
#pragma once
#include "common.cuh"

// x loads: stand-alone kernels read x through the read-only path; inside the persistent kernel x
// was written by other CTAs of the team earlier in the same launch, so it is read with ld.cg (L2).
template <bool RO>
__device__ __forceinline__ double ld_x(const double *p)
{
   if (RO) return __ldg(p);
   // persistent kernel: a plain (L1-cached, coherent-path) load.  Every group barrier ends with __threadfence(), which on
   // sm_100 is MEMBAR.SC.GPU + CCTL.IVALL (the SM's L1 is invalidated), so a line cached before the barrier can never
   // serve a load after it: vectors the group wrote in the previous phase are read fresh, and gathers get L1 reuse.
   // (__ldg / ld.global.nc would be wrong here: the data changes during the launch.)
   return ld_ca(p);
}

// DOT (stand-alone kernels): the fused per-CTA sum of a launch that wants one is sum_i y_i * dw_i instead of sum_i y_i^2 (the
// dot products of the conjugate-gradient solve, pcg.cu).  It is written inline at every row store: routed through a helper
// or a field of SpmvEpilogue, it changed the persistent kernel's spills although that kernel never takes the DOT path.
// DUAL (stand-alone kernels, the same way): a second output y2_i = s2_i * (b_i + y_i) beside y_i.  With the column-scaled
// values and y = b - (A diag(s)) b, y is the t_l of the factorised restriction Rbar_l b = P_l^T t_l and y2 the symmetrised
// smoother's e_l = s o (2b - (A diag(s)) b): one pass over A_l serves both (amgb_options.factor_restriction).

// ---- CSR, LPR lanes per row (vector-per-row; LPR = 32 is warp-per-row) --------------------------
// reference loop: src/SMEM_MatVec.cpp:316-322 (+ the epilogues listed in common.cuh)
template <int LPR, bool RO, bool SVAL, bool DOT = false, bool DUAL = false>
__device__ __forceinline__ double csr_rows_team(const DevCSR &M, const double *__restrict__ x,
                                                double *y, const SpmvEpilogue &e,
                                                int team_tid, int team_size, bool want_sumsq,
                                                const double *dw = nullptr, double *y2 = nullptr, const double *s2 = nullptr)
{
   const int lane = team_tid & (LPR - 1);
   constexpr int RPW = 32 / LPR;                       // rows per warp and iteration
   const int nsub = team_size / LPR;                   // rows per team iteration (multiple of RPW)
   const double *__restrict__ va = SVAL ? M.sval : M.va;
   double sumsq = 0.0;
   // the trip count is uniform per warp so that the full-mask shuffles below are legal
   for (int row0 = (team_tid >> 5) * RPW; row0 < M.nrows; row0 += nsub) {
      const int row = row0 + ((team_tid & 31) / LPR);
      const bool ok = row < M.nrows;
      const int s = ok ? __ldg(M.rp + row) : 0, t = ok ? __ldg(M.rp + row + 1) : 0;
      double acc = 0.0;
      for (int p = s + lane; p < t; p += LPR) acc += ld_stream(va + p) * ld_x<RO>(x + ld_stream(M.ci + p));
      acc = subwarp_sum<LPR>(acc);
      if (lane == 0 && ok) {
         double v = epilogue_apply<RO>(e, row, acc);
         epilogue_store<RO>(e, y, row, v);
         if (want_sumsq) sumsq += DOT ? v * __ldg(dw + row) : v * v;
         if (DUAL) y2[row] = __ldg(s2 + row) * (e.b[row] + v);
      }
   }
   return sumsq;
}

// ---- sliced ELL (C = 32): one thread per row, one warp per slice, coalesced col/val streams -----
// SU == 0: the regular encoding only (the Galerkin / transfer operators: round 1's kernel).
// SU  > 0: the matrix carries the SELL-U encoding (DevCSR::su_desc): a slice is a short list of (delta, mask, value) groups
//          shared by its 32 rows, read SU groups at a time -- the group records (warp-uniform addresses; the lists of a
//          stencil are a few dozen distinct ones, so these are L1 hits), then all x gathers of the batch in flight, then the
//          FMAs.  The descriptor of the warp's NEXT slice is fetched a slice ahead.
// FAST (stand-alone kernels): the warp keeps the DELTAS of the list it met last in registers; consecutive slices of a stencil
//          share one list, so the common slice -- every lane mask full, at most 8 groups -- costs per group one address, one
//          gather, one L1-resident value load and one FMA.  What round 2's measurements say about this kernel family
//          (profiles/README.md R2.3): it is bound by instruction issue and by the number of resident warps, not by HBM --
//          a variant with every value and the epilogue operands held in registers (80 registers, 3 CTAs/SM) was SLOWER
//          (0.226 ms against 0.19) than the generic loop at 56 registers; so this path is written for <= 40 registers.
template <bool RO, bool SVAL, int SU = 0, bool FAST = false, bool DOT = false, bool DUAL = false>
__device__ __forceinline__ double sell_rows_team(const DevCSR &M, const double *__restrict__ x,
                                                 double *y, const SpmvEpilogue &e,
                                                 int team_tid, int team_size, bool want_sumsq, const double *dw = nullptr,
                                                 double *y2 = nullptr, const double *s2 = nullptr)
{
   const int lane = team_tid & 31;
   const int nwarp = team_size >> 5;
   const double *__restrict__ va = SVAL ? M.sell_sval : M.sell_va;
   double sumsq = 0.0;
   int sl = team_tid >> 5;
   int2 dsc = make_int2(0, 0);
   if (SU > 0 && sl < M.sell_slices) dsc = __ldg(M.su_desc + sl);
   int cfirst = -1, ccount = 0;
   bool cfull = false;
   int cd[FAST ? 8 : 1];
   for (; sl < M.sell_slices; sl += nwarp) {
      int row = ((sl + M.sell_base) << 5) + lane;
      if (SU == 0 && M.sell_perm) row = __ldg(M.sell_perm + row);
      double acc = 0.0;
      int2 dnext = make_int2(0, 0);
      if (SU > 0 && sl + nwarp < M.sell_slices) dnext = __ldg(M.su_desc + sl + nwarp);
      if (FAST && dsc.y > 0 && (dsc.x != cfirst || dsc.y != ccount)) {
         cfirst = dsc.x; ccount = dsc.y;
         unsigned int all = 0xffffffffu;
         if (ccount <= 8) {
#pragma unroll
            for (int k = 0; k < 8; k++) {
               const int2 dm = k < ccount ? __ldg(M.su_dm + cfirst + k) : make_int2(0, -1);
               cd[k] = dm.x;
               all &= static_cast<unsigned int>(dm.y);
            }
         } else all = 0u;
         cfull = all == 0xffffffffu;          // every lane takes part in every group (all 32 rows of the slice exist, then)
      }
      if (FAST && dsc.y > 0 && cfull) {
         const double *__restrict__ gv = (SVAL ? M.su_sval : M.su_va) + cfirst;
         const double *__restrict__ xr = x + row;
         double xv[8];
#pragma unroll
         for (int k = 0; k < 8; k++) xv[k] = k < ccount ? ld_x<RO>(xr + cd[k]) : 0.0;
#pragma unroll
         for (int k = 0; k < 8; k++)
            if (k < ccount) acc += __ldg(gv + k) * xv[k];
         const double v = epilogue_apply<RO>(e, row, acc);
         epilogue_store<RO>(e, y, row, v);
         if (want_sumsq) sumsq += DOT ? v * __ldg(dw + row) : v * v;
         if (DUAL) y2[row] = __ldg(s2 + row) * (e.b[row] + v);
      } else if (SU > 0 && dsc.y > 0) {
         const double *__restrict__ gv = SVAL ? M.su_sval : M.su_va;
         const bool ok = row < M.nrows;
         for (int g = 0; g < dsc.y; g += (SU > 0 ? SU : 1)) {
            double xv[SU > 0 ? SU : 1];
            const int2 *__restrict__ dmp = M.su_dm + dsc.x + g;
            const int left = dsc.y - g;
            // all gathers of the batch in flight together; the group VALUES are fetched only when the gathers are back (L1
            // hits), so that nothing but the gathered x occupies registers while the loads are outstanding
#pragma unroll
            for (int k = 0; k < SU; k++) {
               const int2 dm = k < left ? __ldg(dmp + k) : make_int2(0, 0);
               xv[k] = ((static_cast<unsigned int>(dm.y) >> lane) & 1u) ? ld_x<RO>(x + row + dm.x) : 0.0;
            }
#pragma unroll
            for (int k = 0; k < SU; k++)
               if (k < left) acc += __ldg(gv + dsc.x + g + k) * xv[k];
         }
         if (ok) {
            const double v = epilogue_apply<RO>(e, row, acc);
            epilogue_store<RO>(e, y, row, v);
            if (want_sumsq) sumsq += DOT ? v * __ldg(dw + row) : v * v;
            if (DUAL) y2[row] = __ldg(s2 + row) * (e.b[row] + v);
         }
      } else {
         const int off = __ldg(M.sell_off + sl);
         const int width = (__ldg(M.sell_off + sl + 1) - off) >> 5;
         const int *__restrict__ cp = M.sell_ci + off + lane;
         const double *__restrict__ vp = va + off + lane;
#pragma unroll 4
         for (int k = 0; k < width; k++) acc += ld_stream(vp + (k << 5)) * ld_x<RO>(x + ld_stream(cp + (k << 5)));
         if (row >= 0 && row < M.nrows) {
            double v = epilogue_apply<RO>(e, row, acc);
            epilogue_store<RO>(e, y, row, v);
            if (want_sumsq) sumsq += DOT ? v * __ldg(dw + row) : v * v;
            if (DUAL) y2[row] = __ldg(s2 + row) * (e.b[row] + v);
         }
      }
      dsc = dnext;
   }
   return sumsq;
}

// ---- SELL-C-sigma with the epilogue applied in row order (stand-alone kernel only) ---------------
// Inside a window of sigma rows the rows are sorted by length, so in sell_rows_team lane l of a slice owns a row scattered over
// the window, and every epilogue load and store is a warp access spread over up to 8 lines.  Here a CTA of NT threads takes the
// NT / 32 consecutive slices [s0, s0 + NT / 32) per iteration: when sigma divides NT and the view starts at a multiple of
// NT / 32 slices, their slots hold exactly the rows [32 (s0 + sell_base), + NT) (launch_spmv checks that).  Each lane sums
// its row as sell_rows_team does (same entries, same order), parks the sum in shared memory at the row's place, and after a
// barrier thread t applies the unchanged epilogue to the t-th row of the range: the epilogue's loads and stores are coalesced.
// The trip count is CTA-uniform, so every thread reaches every barrier; the two halves of `sacc` ([2 * NT]) alternate, so one
// barrier per iteration separates the writes of an iteration from the reads of the one before.
template <int NT, bool SVAL, bool DOT = false, bool DUAL = false>
__device__ __forceinline__ double sell_window_rows_cta(const DevCSR &M, const double *__restrict__ x, double *y,
                                                       const SpmvEpilogue &e, bool want_sumsq, const double *dw, double *y2,
                                                       const double *s2, double *sacc)
{
   constexpr int SPC = NT / 32;                        // slices per CTA and iteration
   const int lane = threadIdx.x & 31;
   const double *__restrict__ va = SVAL ? M.sell_sval : M.sell_va;
   double sumsq = 0.0;
   double *buf = sacc;
   for (int s0 = blockIdx.x * SPC; s0 < M.sell_slices; s0 += gridDim.x * SPC) {
      const int sl = s0 + (threadIdx.x >> 5);
      const int base = (s0 + M.sell_base) << 5;        // first slot of the CTA's slices = first row of its windows
      if (sl < M.sell_slices) {
         const int row = __ldg(M.sell_perm + base + threadIdx.x);
         const int off = __ldg(M.sell_off + sl);
         const int width = (__ldg(M.sell_off + sl + 1) - off) >> 5;
         const int *__restrict__ cp = M.sell_ci + off + lane;
         const double *__restrict__ vp = va + off + lane;
         double acc = 0.0;
#pragma unroll 4
         for (int k = 0; k < width; k++) acc += ld_stream(vp + (k << 5)) * ld_x<true>(x + ld_stream(cp + (k << 5)));
         if (row >= 0 && row < M.nrows) buf[row - base] = acc;
      }
      __syncthreads();
      const int row = base + threadIdx.x;
      if (row < M.nrows) {
         const double v = epilogue_apply<true>(e, row, buf[threadIdx.x]);
         epilogue_store<true>(e, y, row, v);
         if (want_sumsq) sumsq += DOT ? v * __ldg(dw + row) : v * v;
         if (DUAL) y2[row] = __ldg(s2 + row) * (e.b[row] + v);
      }
      buf = buf == sacc ? sacc + NT : sacc;
   }
   return sumsq;
}

// ---- warp-stream: CSR row chunks at warp granularity, no CTA-wide barriers -----------------------
// Every WARP owns every team_nwarps-th row chunk (DevCSR::blk, <= AMGB_WARP_CHUNK entries).
// Lanes load the chunk's (col,val) pairs coalesced (consecutive lanes = consecutive entries, all 2*EPT
// loads issued before the first use), gather x, park the products in the warp's private slice of shared
// memory, __syncwarp, and sum each row with a sub-warp sized to the chunk's row count.  Warps never wait
// for each other, so the load / gather / reduce phases of the 32-64 resident warps of an SM overlap
// freely -- a CTA-synchronous form of the same idea spent ~20 % of its issue slots in barrier stalls and ~45 %
// waiting on gathers with only 3-5 CTAs to hide them (DESIGN.md 3.3).  swarp: AMGB_WARP_CHUNK doubles per warp.
template <bool RO, bool SVAL, bool DOT = false, bool DUAL = false>
__device__ __forceinline__ double warp_stream_rows_team(const DevCSR &M, const double *__restrict__ x, double *y,
                                                        const SpmvEpilogue &e, int team_warp, int team_nwarps,
                                                        double *swarp, bool want_sumsq, const double *dw = nullptr,
                                                        double *y2 = nullptr, const double *s2 = nullptr)
{
   constexpr int CAP = AMGB_WARP_CHUNK, EPT = CAP / 32;
   const int lane = threadIdx.x & 31;
   const double *__restrict__ va = SVAL ? M.sval : M.va;
   double sumsq = 0.0;
   int4 d = team_warp < M.nblk ? __ldg(M.blk + team_warp) : make_int4(0, 0, 0, 0);
   for (int b = team_warp; b < M.nblk; b += team_nwarps) {
      const int r0 = d.x, r1 = d.y, p0 = d.z, p1 = d.w, nr = r1 - r0, cnt = p1 - p0;
      if (b + team_nwarps < M.nblk) d = __ldg(M.blk + b + team_nwarps);
      if (cnt > CAP) {
         // a single long row: the warp strides over it
         double acc = 0.0;
         for (int p = p0 + lane; p < p1; p += 32) acc += ld_stream(va + p) * ld_x<RO>(x + ld_stream(M.ci + p));
         acc = subwarp_sum<32>(acc);
         if (lane == 0) {
            const double v = epilogue_apply<RO>(e, r0, acc);
            y[r0] = v;
            if (want_sumsq) sumsq += DOT ? v * __ldg(dw + r0) : v * v;
            if (DUAL) y2[r0] = __ldg(s2 + r0) * (e.b[r0] + v);
         }
         continue;
      }
      int cc[EPT];
      double vv[EPT];
      const int *__restrict__ ci = M.ci;               // (read through M.ci directly, ptxas lays the long-row branch out differently)
#pragma unroll
      for (int k = 0; k < EPT; k++) {
         const int q = lane + 32 * k;
         cc[k] = 0; vv[k] = 0.0;
         if (q < cnt) {
            cc[k] = ld_stream(ci + p0 + q);
            vv[k] = ld_stream(va + p0 + q);
         }
      }
      // lanes per row: the largest power of two such that all rows fit in one pass
      int lpr = 1;
      while (lpr < 32 && nr * (lpr << 1) <= 32) lpr <<= 1;
      const int sub = lane & (lpr - 1);
      const int row_a = r0 + lane / lpr;
      const bool ok_a = row_a < r1;
      int s_a = 0, t_a = 0;
      EpiOps o_a;
         o_a.b = 0.0; o_a.c = 0.0; o_a.rs = 1.0;
      if (ok_a) {
         s_a = __ldg(M.rp + row_a) - p0;
         t_a = __ldg(M.rp + row_a + 1) - p0;
         if (sub == 0) o_a = epilogue_load<RO>(e, row_a);
      }
#pragma unroll
      for (int k = 0; k < EPT; k++) {
         const int q = lane + 32 * k;
         if (q < cnt) vv[k] *= ld_x<RO>(x + cc[k]);
      }
      __syncwarp();                                    // the previous chunk's readers are done
#pragma unroll
      for (int k = 0; k < EPT; k++) {
         const int q = lane + 32 * k;
         if (q < cnt) swarp[q] = vv[k];
      }
      __syncwarp();
      {
         double acc = 0.0;
         for (int q = s_a + sub; q < t_a; q += lpr) acc += swarp[q];
         for (int o = lpr >> 1; o > 0; o >>= 1) acc += __shfl_down_sync(AMGB_FULL, acc, o, 32);
         if (sub == 0 && ok_a) {
            const double v = epilogue_finish(e, o_a, acc);
            y[row_a] = v;
            if (want_sumsq) sumsq += DOT ? v * __ldg(dw + row_a) : v * v;
            if (DUAL) y2[row_a] = __ldg(s2 + row_a) * (e.b[row_a] + v);
         }
      }
      for (int base = 32; base < nr; base += 32) {     // only when lpr == 1
         const int row = r0 + base + lane;
         if (row < r1) {
            const int s1 = __ldg(M.rp + row) - p0, t1 = __ldg(M.rp + row + 1) - p0;
            double acc = 0.0;
            for (int q = s1; q < t1; q++) acc += swarp[q];
            const double v = epilogue_apply<RO>(e, row, acc);
            y[row] = v;
            if (want_sumsq) sumsq += DOT ? v * __ldg(dw + row) : v * v;
            if (DUAL) y2[row] = __ldg(s2 + row) * (e.b[row] + v);
         }
      }
   }
   return sumsq;
}

// vector-per-row CSR with the lanes-per-row chosen at upload time
template <bool RO, bool SVAL, bool DOT = false, bool DUAL = false>
__device__ __forceinline__ double csr_rows_dispatch(const DevCSR &M, const double *x, double *y, const SpmvEpilogue &e,
                                                    int team_tid, int team_size, bool want_sumsq, const double *dw = nullptr,
                                                 double *y2 = nullptr, const double *s2 = nullptr)
{
   switch (M.lpr) {
      case 2: return csr_rows_team<2, RO, SVAL, DOT, DUAL>(M, x, y, e, team_tid, team_size, want_sumsq, dw, y2, s2);
      case 4: return csr_rows_team<4, RO, SVAL, DOT, DUAL>(M, x, y, e, team_tid, team_size, want_sumsq, dw, y2, s2);
      case 8: return csr_rows_team<8, RO, SVAL, DOT, DUAL>(M, x, y, e, team_tid, team_size, want_sumsq, dw, y2, s2);
      case 16: return csr_rows_team<16, RO, SVAL, DOT, DUAL>(M, x, y, e, team_tid, team_size, want_sumsq, dw, y2, s2);
      default: return csr_rows_team<32, RO, SVAL, DOT, DUAL>(M, x, y, e, team_tid, team_size, want_sumsq, dw, y2, s2);
   }
}


// ---- hybrid Jacobi / Gauss-Seidel (src/SMEM_Smooth.cpp:533-586) ----------------------------------
// Gauss-Seidel inside a block of `B` consecutive rows (one thread walks one block in row order),
// Jacobi across blocks.  Zero-guess form (:549-562): out-of-block terms are skipped.  General form
// (:565-581): in-block columns read live u, others u_prev.  Divisor a_ii (weight forced to 1,
// :546) unless `scale` (= a_ii/omega, Parfor variant :253-263) is given.
template <bool RO>
__device__ __forceinline__ void hybrid_jgs_team(const DevCSR &A, const double *__restrict__ f,
                                                double *u, const double *__restrict__ u_prev,
                                                const double *__restrict__ scale, int B, bool zero_guess,
                                                int team_tid, int team_size)
{
   const int nblocks = (A.nrows + B - 1) / B;
   for (int blk = team_tid; blk < nblocks; blk += team_size) {
      const int ns = blk * B, ne = min(ns + B, A.nrows);
      if (zero_guess)
         for (int i = ns; i < ne; i++) u[i] = 0.0;
      for (int i = ns; i < ne; i++) {
         const int s = A.rp[i], t = A.rp[i + 1];
         const double d = A.va[s];
         if (d != 0.0) {
            double res = ld_x<RO>(f + i);
            for (int p = s; p < t; p++) {
               const int ii = A.ci[p];
               if (ii >= ns && ii < ne) res -= A.va[p] * u[ii];
               else if (!zero_guess) res -= A.va[p] * ld_x<RO>(u_prev + ii);
            }
            const double div = scale ? scale[i] : d;
            if (zero_guess) u[i] = res / div;
            else u[i] += res / div;
         }
      }
   }
}

// ---- hybrid JGS, sub-warp per block --------------------------------------------------------------
// The same sweep with LPB lanes cooperating on one block: the block's rows are visited in order (that is the
// Gauss-Seidel dependence), but each row's dot product is spread over the LPB lanes (coalesced entry loads, a
// shuffle reduction) and the block's live u values sit in the sub-warp's slice of shared memory.  With one
// THREAD per block (hybrid_jgs_team) every load of the sweep is an uncoalesced dependent access: 1.9 ms on the
// 256^3 fine level against 0.32 ms for a Jacobi sweep, and hundreds of microseconds on coarse levels that have
// a handful of blocks.  ub: AMGB_JGS_BMAX doubles per sub-warp; requires B <= AMGB_JGS_BMAX.
#define AMGB_JGS_BMAX 64
template <bool RO, int LPB>
__device__ __forceinline__ void hybrid_jgs_subwarp_team(const DevCSR &A, const double *__restrict__ f, double *u,
                                                        const double *__restrict__ u_prev, const double *__restrict__ scale,
                                                        int B, bool zero_guess, int team_tid, int team_size, double *smem_u)
{
   const int lane = team_tid & (LPB - 1);
   double *ub = smem_u + (threadIdx.x / LPB) * AMGB_JGS_BMAX;
   const int nblocks = (A.nrows + B - 1) / B;
   const int nsw = team_size / LPB;                     // sub-warps in the team
   // the trip count is uniform per warp (full-mask shuffles below)
   for (int blk0 = (team_tid >> 5) * (32 / LPB); blk0 < nblocks; blk0 += nsw) {
      const int blk = blk0 + ((team_tid & 31) / LPB);
      const bool active = blk < nblocks;
      const int ns = blk * B, ne = active ? min(ns + B, A.nrows) : ns;
      for (int i = lane; i < B; i += LPB) ub[i] = (!zero_guess && ns + i < ne) ? (RO ? u[ns + i] : ld_cg(u + ns + i)) : 0.0;
      __syncwarp();
      for (int r = 0; r < B; r++) {
         const int row = ns + r;
         const bool ok = row < ne;
         const int s = ok ? __ldg(A.rp + row) : 0, t = ok ? __ldg(A.rp + row + 1) : 0;
         double acc = 0.0;
         for (int p = s + lane; p < t; p += LPB) {
            const int ii = ld_stream(A.ci + p);
            if (ii >= ns && ii < ne) acc += ld_stream(A.va + p) * ub[ii - ns];
            else if (!zero_guess) acc += ld_stream(A.va + p) * ld_x<RO>(u_prev + ii);
         }
#pragma unroll
         for (int o = LPB >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(AMGB_FULL, acc, o);
         if (lane == 0 && ok && t > s) {
            const double d = __ldg(A.va + s);
            if (d != 0.0) {
               const double res = ld_x<RO>(f + row) - acc;
               const double div = scale ? __ldg(scale + row) : d;
               ub[r] = zero_guess ? res / div : ub[r] + res / div;
            }
         }
         __syncwarp();
      }
      for (int i = lane; i < B; i += LPB)
         if (ns + i < ne) u[ns + i] = ub[i];
      __syncwarp();
   }
}

// ---- (semi-)asynchronous Gauss-Seidel (src/SMEM_Smooth.cpp:445-502) -------------------------------
// Every thread sweeps its blocks of `B` consecutive rows in order, reading whatever the other threads have
// written to u so far (chaotic relaxation): u_i += (f_i - sum_j a_ij u_j) / a_ii.  The asynchronous variant
// runs all `sweeps` without synchronising; the semi-asynchronous one is launched once per sweep (the kernel
// boundary is its barrier).  u is read and written through L2 (ld.cg / st.cg) so that updates become visible.
template <bool RO>
__device__ __forceinline__ void async_gs_team(const DevCSR &A, const double *__restrict__ f, double *u, int B, int sweeps,
                                              int team_tid, int team_size)
{
   const int nblocks = (A.nrows + B - 1) / B;
   for (int k = 0; k < sweeps; k++)
      for (int blk = team_tid; blk < nblocks; blk += team_size) {
         const int ns = blk * B, ne = min(ns + B, A.nrows);
         for (int i = ns; i < ne; i++) {
            const int s = A.rp[i], t = A.rp[i + 1];
            const double d = A.va[s];
            if (d != 0.0) {
               double res = ld_x<RO>(f + i);
               for (int p = s; p < t; p++) res -= A.va[p] * ld_cg(u + A.ci[p]);
               st_cg(u + i, ld_cg(u + i) + res / d);
            }
         }
      }
}

// ---- y += M^T x (SMEM_MatVecT / SMEM_Restrict with -no_construct_R, src/SMEM_MatVec.cpp:325-408) --------
// LPR lanes walk one row of M and scatter its contributions with fp64 reductions; y must be zeroed first.
template <int LPR>
__device__ __forceinline__ void csr_transpose_rows_team(const DevCSR &M, const double *__restrict__ x, double *y,
                                                        int team_tid, int team_size)
{
   const int lane = team_tid & (LPR - 1);
   for (int row = team_tid / LPR; row < M.nrows; row += team_size / LPR) {
      const double xr = __ldg(x + row);
      const int s = __ldg(M.rp + row), t = __ldg(M.rp + row + 1);
      for (int p = s + lane; p < t; p += LPR) red_add_f64(y + ld_stream(M.ci + p), ld_stream(M.va + p) * xr);
   }
}

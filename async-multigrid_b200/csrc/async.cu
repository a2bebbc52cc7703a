// async.cu -- the asynchronous additive AMG solve as ONE persistent cooperative kernel.
//
// Replaces SMEM_Async_Add_AMG (src/SMEM_Async_AMG.cpp:7-437).  The reference runs one long-lived
// OpenMP parallel region in which every AMG level owns a group of threads; a group loops
//   restrict chain -> smooth on its level -> prolong chain -> atomic add into the shared u ->
//   private copy of u -> private residual r = f - A u_private
// with barriers only INSIDE the group (SMEM_LevelBarrier, src/Misc.cpp:485-533) and no barrier
// between groups.  Here a group is a contiguous range of CTAs of a cooperative launch (all CTAs
// co-resident, so the spin barriers make progress); the shared u is updated with red.global.add.f64;
// the group barrier is an arrive counter + generation word in global memory.
//
// Round-2 design: the kernel is an INTERPRETER of per-group programs (launch.h AsyncOp).  Round 1's kernel inlined
// every chain with a CTA-synchronous, TMA-staged SpMV: 80 registers, 3 CTAs per SM, 37 % of the warp slots -- ncu
// (profiles/r2_ncu_full_async_kernel_r1design.csv) shows it latency-bound at 30 % of DRAM throughput with barrier and
// scoreboard stalls, not starved for instructions.  This kernel has ONE SpMV call site built from the same
// occupancy-friendly pieces as the stand-alone kernels (sliced ELL incl. SELL-U and SELL-C-sigma, vector-per-row CSR),
// L1-cached gathers (see ld_x<false>), fused "u += e; u_k = u" epilogues, and the level-0 transfers in factorised form.
// Termination mirrors the reference: LOCAL = a group stops after num_cycles own corrections
// (:317-322); GLOBAL = the finest group's root raises converge_flag once every level has done num_cycles
// (CheckConverge, src/Misc.cpp:418-442) and every group sees it at its next barrier (:323-337).
#include "ctx.h"
#include "kernels.cuh"
#include "async_team.cuh"
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

namespace {

__device__ __forceinline__ unsigned long long global_ns()
{
   unsigned long long t;
   asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
   return t;
}

// The current operation and the matrix view it works on live in SHARED memory: every thread reads the fields it needs where
// it needs them (the stand-alone kernels get them from the constant bank), so neither the epilogue nor the matrix
// descriptor is held in registers across the SpMV loops -- that is what keeps this kernel at 40 registers, 6 CTAs per SM.
struct OpView {
   AsyncOp op;
   DevCSR M;
};

// thread 0: the view of the operator this CTA works on -- the column-scaled values when asked for, and, for a CTA-slice
// operation, this CTA's share of the rows, the rows of level 0 being dealt to the CTAs of all WORKING groups (the
// reference deals them to all threads, A_ns_global / A_ne_global, src/SMEM_Setup.cpp:923-939; the idle coarsest group is
// left out here: it finishes its num_cycles empty iterations at once, and the rows of a group that has stopped are
// never smoothed or refreshed again): whole slices of a sliced-ELL operator, else rows
__device__ __forceinline__ void make_view(OpView &v, const DevCSR &M0, int slice_ctas)
{
   v.M = M0;
   DevCSR &M = v.M;
   if (v.op.sval) { M.va = M0.sval; M.sell_va = M0.sell_sval; M.su_va = M0.su_sval; }
   if (!v.op.range) return;
   const long units = M.sell_slices > 0 ? M.sell_slices : M.nrows;
   const long cta = min((long)blockIdx.x, (long)slice_ctas);      // (a CTA beyond slice_ctas -- the idle coarsest group -- gets nothing)
   const int u0 = (int)(units * cta / slice_ctas), u1 = (int)(units * min(cta + 1, (long)slice_ctas) / slice_ctas);
   if (M.sell_slices > 0) {
      M.sell_off += u0; M.sell_base += u0; M.sell_slices = u1 - u0;
      if (M.su_desc) M.su_desc += u0;
   } else {
      SpmvEpilogue &e = v.op.e;
      M.rp += u0; M.nrows = u1 - u0;
      if (v.op.y) v.op.y += u0;
      if (e.b) e.b += u0;
      if (e.c) e.c += u0;
      if (e.rs) e.rs += u0;
      if (e.b2) e.b2 += u0;
      if (e.xs) e.xs += u0;
      if (e.red) e.red += u0;
      if (e.red_copy) e.red_copy += u0;
      if (e.acc) e.acc += u0;
   }
}

// this CTA's row range when level-0 rows are dealt to all CTAs (matches make_view)
__device__ __forceinline__ void cta_slice_rows(const DevCSR &M, int slice_ctas, int *r0, int *r1)
{
   const long units = M.sell_slices > 0 ? M.sell_slices : M.nrows;
   const long cta = min((long)blockIdx.x, (long)slice_ctas);
   const long u0 = units * cta / slice_ctas, u1 = units * min(cta + 1, (long)slice_ctas) / slice_ctas;
   if (M.sell_slices > 0) { *r0 = (int)min((long)M.nrows, u0 * 32); *r1 = (int)min((long)M.nrows, u1 * 32); }
   else { *r0 = (int)u0; *r1 = (int)u1; }
}

// EXT: the instantiation of the asynchronous implicit extended-system solver (extended.cu): the AOP_EXT_* operations, a
// per-CTA omega / loc_iters, and an L1 invalidation after the barrier of a one-CTA group too (its reads of other groups'
// u_j / e_j must never be served by a line cached before the barrier).  HEAVY = false / EXT = false and HEAVY = true are the
// asynchronous additive solver's instantiations; the EXT branches compile out of them.
template <bool HEAVY, bool EXT = false>
__global__ void __launch_bounds__(kABlock, HEAVY ? 3 : 6) k_async_amg(const AsyncParams *__restrict__ pp)
{
   const AsyncParams &p = *pp;
   const int L = p.num_levels;
   // which level's group does this CTA belong to
   int q = p.first_group;
   while (q + 1 < L && (int)blockIdx.x >= p.cta_begin[q + 1]) q++;
   Team tm;
   tm.cta = blockIdx.x - p.cta_begin[q];
   tm.nctas = p.cta_begin[q + 1] - p.cta_begin[q];
   tm.tid = tm.cta * kABlock + threadIdx.x;
   tm.size = tm.nctas * kABlock;
   tm.count = p.barrier_count + q;
   tm.gen = p.barrier_gen + q;
   extern __shared__ __align__(16) unsigned char dyn_smem[];   // HEAVY only: the hybrid-JGS sub-warps' live block values
   tm.smem = dyn_smem;
   __shared__ int s_stop;
   __shared__ __align__(16) unsigned char sv_raw[sizeof(OpView)];   // (raw bytes: the structs carry default member initialisers)
   OpView &sv = *reinterpret_cast<OpView *>(sv_raw);
   const AsyncOp *prog = p.ops + p.op_begin[q];
   const int nops = p.op_begin[q + 1] - p.op_begin[q];
   const unsigned long long t_begin = global_ns();
   int stop = 0;
   unsigned long long seq = 0;            // exchange steps of this group so far (row-partitioned solve)
   double omega = 2.0;                    // EXT: the group's Chebyshev omega, advanced identically by every CTA of the group
   int loc_iters = 1;                     // EXT: the group's loc_iters (every CTA keeps the same count)

   while (!stop) {
      for (int i = 0; i < nops; i++) {
         __syncthreads();                              // the previous operation's readers are done with sv
         if (threadIdx.x < (int)(sizeof(AsyncOp) / sizeof(int)))
            reinterpret_cast<int *>(&sv.op)[threadIdx.x] = __ldg(reinterpret_cast<const int *>(prog + i) + threadIdx.x);
         __syncthreads();
         const AsyncOp &op = sv.op;
         const int type = op.type;
         if (type == AOP_SPMV || (EXT && type == AOP_EXT_RESID)) {
            if (threadIdx.x == 0)
               make_view(sv, op.mat_kind == AMGB_MAT_A ? p.A[op.mat_level] : (op.mat_kind == AMGB_MAT_P ? p.P[op.mat_level] : (op.mat_kind == AMGB_MAT_R ? p.R[op.mat_level] : p.Ainv)), p.slice_ctas);
            __syncthreads();
            const DevCSR &M = sv.M;
            const int t0 = op.range ? (int)threadIdx.x : tm.tid, ts = op.range ? kABlock : tm.size;
            const bool ss = EXT && type == AOP_EXT_RESID;
            double part = 0.0;
            if (M.sell_slices > 0 && M.su_desc) part = sell_rows_team<false, false, 4>(M, op.x, op.y, op.e, t0, ts, ss);
            else if (M.sell_slices > 0) part = sell_rows_team<false, false>(M, op.x, op.y, op.e, t0, ts, ss);
            else if (M.nrows > 0) part = csr_rows_dispatch<false, false>(M, op.x, op.y, op.e, t0, ts, ss);
            if (ss) {
               part = block_sum(part);
               if (threadIdx.x == 0) *((volatile double *)(p.ext.cta_ss + blockIdx.x)) = part;
            }
         } else if (EXT && type == AOP_EXT_CHEBY) {
            // u_k <- y_k + omega (delta rs o r_k + u_k - y_k), y_k <- old u_k (k_cheby's arithmetic).  u_k is read by the other
            // groups while this runs: stored through L2
            const int n = p.A[op.level].nrows;
            const double dl = p.ext.delta;
            for (int k = tm.tid; k < n; k += tm.size) {
               const double uo = ld_cg(op.y + k), yo = ld_cg(op.e.c + k);
               const double s = __ldg(op.e.rs + k) * ld_cg(op.x + k);
               st_cg(op.y + k, yo + omega * (dl * s + uo - yo));
               st_cg(const_cast<double *>(op.e.c) + k, uo);
            }
            omega = 1.0 / (1.0 - omega / p.ext.mu22);
         } else if (EXT && type == AOP_EXT_STOP) {
            // the stop rule of SMEM_ExtendedSystemSolve's asynchronous branch (src/SMEM_ExtendedSystem.cpp:636-652); the previous
            // operation's barrier made every CTA's residual slot visible
            if (tm.tid == 0) {
               double s = 0.0;
               for (int t = p.cta_begin[q]; t < p.cta_begin[q + 1]; t++) s += *((volatile double *)(p.ext.cta_ss + t));
               if (loc_iters > 1) p.ext.contrib[q] = s;         // check_resnorm_flag && loc_iters > 1, before the increment
               __threadfence();
               if (q == 0 && *p.converge_flag == 0) {           // the reference's thread 0: sum of the (possibly stale) contributions
                  double tot = 0.0;
                  for (int l = 0; l < L; l++) tot += p.ext.contrib[l];
                  if (sqrt(tot) / p.ext.r0_ext < p.ext.tol) { *p.converge_flag = 1; __threadfence(); }
               }
               if (loc_iters + 1 == p.num_cycles) { atomicAdd(p.ext.done, 1); __threadfence(); }
               const int st = *p.converge_flag != 0 || *((volatile int *)p.ext.done) >= L;
               *((volatile int *)(p.group_stop + q)) = st;
               if (tm.nctas == 1) s_stop = st;
            }
            loc_iters++;
            // every CTA takes the group root's decision
            if (tm.nctas > 1) {
               group_barrier(tm);
               if (threadIdx.x == 0) s_stop = *((volatile int *)(p.group_stop + q));
            }
            __syncthreads();
            stop = s_stop;
            __syncthreads();
         } else if (type == AOP_SCALE) {
            // y = rs o x (zero-guess Jacobi, src/SMEM_Smooth.cpp:381-389), optionally reduced into the shared u
            int r0 = 0, r1 = p.A[op.level].nrows, step = tm.size, first = tm.tid;
            if (op.range) { cta_slice_rows(p.A[op.level], p.slice_ctas, &r0, &r1); step = kABlock; first = threadIdx.x; }
            for (int k = r0 + first; k < r1; k += step) {
               const double v = __ldg(op.e.rs + k) * ld_cg(op.x + k);
               if (op.e.red) {
                  red_add_f64(op.e.red + k, v);
                  if (op.e.red_copy) op.e.red_copy[k] = ld_cg(op.e.red + k);
               }
               if (op.y) op.y[k] = v;
            }
         } else if (type == AOP_COPY) {
            const int n = p.A[op.level].nrows;
            for (int k = tm.tid; k < n; k += tm.size) op.y[k] = ld_cg(op.x + k);
         } else if (type == AOP_ZERO) {
            const int n = p.A[op.level].nrows;
            for (int k = tm.tid; k < n; k += tm.size) st_cg(op.y + k, 0.0);
         } else if (type == AOP_UPDATE) {
            // u += e, private copy (src/SMEM_Async_AMG.cpp:285-301); `locked`: plain read-modify-write inside the
            // SEMI_ASYNC critical section (:238-283); acc: the group's accumulated correction (-read_type res)
            const int n = p.n0;
            double *tgt = op.e.red, *cp = op.e.red_copy, *acc = op.e.acc;
            for (int k = tm.tid; k < n; k += tm.size) {
               const double ev = ld_cg(op.x + k);
               if (acc) acc[k] += ev;
               if (!tgt) continue;
               if (op.locked) {
                  const double v = ld_cg(tgt + k) + op.e.red_scale * ev;
                  st_cg(tgt + k, v);
                  if (cp) cp[k] = v;
               } else {
                  red_add_f64(tgt + k, op.e.red_scale * ev);
                  if (cp) cp[k] = ld_cg(tgt + k);
               }
            }
         } else if (type == AOP_PUSH) {
            // row-partitioned solve: this group's boundary (or owned) entries of a vector go straight into the ghost slots
            // of the same group's vector on a peer GPU -- plain stores over NVLink, nobody waits for them (dist_async.cu)
            const int n = op.sweeps;
            for (int k = tm.tid; k < n; k += tm.size) op.y[k] = ld_cg(op.x + k);
            __threadfence_system();
         } else if (type == AOP_SIGNAL) {
            // exchange step `seq` of this group: once every CTA's stores are fenced and done, the group root publishes the
            // step number in the peer's flag word (release at system scope)
            if (op.zero) { group_barrier(tm); seq++; }
            if (tm.tid == 0 && op.y) {
               __threadfence_system();
               *reinterpret_cast<volatile unsigned long long *>(op.y) = seq;
            }
         } else if (type == AOP_WAIT) {
            // ... and waits for the same step from the peer (the same group there runs the same program).  Bounded: a peer that
            // never arrives (its launch failed) must end this kernel with an error, not hang the GPU.
            if (tm.tid == 0 && op.x) {
               const volatile unsigned long long *flag = reinterpret_cast<const volatile unsigned long long *>(op.x);
               const unsigned long long t_wait = global_ns();
               while (*flag < seq && p.converge_flag[1] == 0) {      // (after one time-out nobody waits any more: the launch just ends)
                  __nanosleep(128);
                  if (global_ns() - t_wait > 30000000000ull) { p.converge_flag[1] = 1; __threadfence(); break; }
               }
               __threadfence_system();
            }
            if (op.barrier) {
               // every CTA drops what its SM's L1 holds of the ghost slots (a one-CTA group's barrier has no fence of its own)
               group_barrier(tm);
               if (threadIdx.x == 0) __threadfence();
               __syncthreads();
            }
         } else if (type == AOP_LOCK) {
            if (tm.tid == 0) {
               while (atomicCAS(p.lock, 0, 1) != 0) __nanosleep(64);
               __threadfence();
            }
         } else if (type == AOP_UNLOCK) {
            if (tm.tid == 0) {
               __threadfence();
               atomicExch(p.lock, 0);
            }
         } else if (type == AOP_COUNT_STOP) {
            // correction count and stop rule (:314-337)
            if (tm.tid == 0) {
               const int cnt = *((volatile int *)(p.num_correct + q)) + 1;
               *((volatile int *)(p.num_correct + q)) = cnt;
               __threadfence();
               if (p.converge_type == AMGB_CONVERGE_GLOBAL && q == p.first_group && *p.converge_flag == 0) {
                  int all = 1;
                  for (int l = p.first_group; l < L; l++)
                     if (*((volatile int *)(p.num_correct + l)) < p.num_cycles) { all = 0; break; }
                  if (all) { *p.converge_flag = 1; __threadfence(); }
               }
            }
            group_barrier(tm);
            if (threadIdx.x == 0) {
               int st;
               if (p.converge_type == AMGB_CONVERGE_LOCAL) st = *((volatile int *)(p.num_correct + q)) >= p.num_cycles;
               else st = *p.converge_flag;
               s_stop = st;
            }
            // all CTAs of the group must take the same decision: publish the root CTA's view
            if (tm.nctas > 1 && p.converge_type != AMGB_CONVERGE_LOCAL) {
               // GLOBAL: the flag may flip between two CTAs' reads; the group root decides
               __syncthreads();
               if (tm.cta == 0 && threadIdx.x == 0) { *((volatile int *)(p.group_stop + q)) = s_stop; __threadfence(); }
               group_barrier(tm);
               if (threadIdx.x == 0) s_stop = *((volatile int *)(p.group_stop + q));
            }
            __syncthreads();
            stop = s_stop;
            __syncthreads();
         } else if (HEAVY && type == AOP_JGS) {
            const DevCSR &A = p.A[op.level];
            double *su = reinterpret_cast<double *>(tm.smem);
            const bool zero = op.zero != 0;
            switch (p.jgs_lpb[op.level]) {   // sub-warp per block (see hybrid_jgs_subwarp_team); 0: block longer than the staging slice
               case 4: hybrid_jgs_subwarp_team<false, 4>(A, op.x, op.y, op.e.c, nullptr, p.jgs_block_rows, zero, tm.tid, tm.size, su); break;
               case 8: hybrid_jgs_subwarp_team<false, 8>(A, op.x, op.y, op.e.c, nullptr, p.jgs_block_rows, zero, tm.tid, tm.size, su); break;
               case 16: hybrid_jgs_subwarp_team<false, 16>(A, op.x, op.y, op.e.c, nullptr, p.jgs_block_rows, zero, tm.tid, tm.size, su); break;
               case 32: hybrid_jgs_subwarp_team<false, 32>(A, op.x, op.y, op.e.c, nullptr, p.jgs_block_rows, zero, tm.tid, tm.size, su); break;
               default: hybrid_jgs_team<false>(A, op.x, op.y, op.e.c, nullptr, p.jgs_block_rows, zero, tm.tid, tm.size);
            }
         } else if (HEAVY && type == AOP_ASYNC_GS) {
            async_gs_team<false>(p.A[op.level], op.x, op.y, p.jgs_block_rows, op.sweeps, tm.tid, tm.size);
         }
         if (op.barrier && type != AOP_WAIT) group_barrier(tm);
         if (EXT && op.barrier && tm.nctas == 1) {
            // (a one-CTA group's barrier has no fence of its own: drop what this SM's L1 holds of the other groups' vectors)
            if (threadIdx.x == 0) __threadfence();
            __syncthreads();
         }
      }
   }
   if (tm.tid == 0) p.group_ns[q] = global_ns() - t_begin;
   if (EXT && tm.tid == 0) p.ext.loc_iters[q] = loc_iters;
}

constexpr size_t kHeavySmem = (size_t)(kABlock / 4) * AMGB_JGS_BMAX * sizeof(double);

}  // namespace

int async_max_grid(int block, bool heavy)
{
   int dev = 0, sms = 0, per_sm = 0;
   cudaGetDevice(&dev);
   cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
   if (heavy) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_async_amg<true>, block, kHeavySmem);
   else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_async_amg<false>, block, 0);
   return sms * per_sm;
}

int launch_async(cudaStream_t st, const AsyncParams *params_dev, int grid, int block, bool heavy, const cudaAccessPolicyWindow *window)
{
   cudaLaunchConfig_t cfg = {};
   cfg.gridDim = dim3(grid);
   cfg.blockDim = dim3(block);
   cfg.dynamicSmemBytes = heavy ? kHeavySmem : 0;
   cfg.stream = st;
   cudaLaunchAttribute attrs[2];
   int na = 0;
   attrs[na].id = cudaLaunchAttributeCooperative;
   attrs[na].val.cooperative = 1;
   na++;
   if (window && window->num_bytes > 0) {
      attrs[na].id = cudaLaunchAttributeAccessPolicyWindow;
      attrs[na].val.accessPolicyWindow = *window;
      na++;
   }
   cfg.attrs = attrs;
   cfg.numAttrs = na;
   cudaError_t e = heavy ? cudaLaunchKernelEx(&cfg, k_async_amg<true>, params_dev) : cudaLaunchKernelEx(&cfg, k_async_amg<false>, params_dev);
   return e == cudaSuccess ? 1 : -(int)e;
}

int async_max_grid_ext(int block)
{
   int dev = 0, sms = 0, per_sm = 0;
   cudaGetDevice(&dev);
   cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
   cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_async_amg<false, true>, block, 0);
   return sms * per_sm;
}

int launch_async_ext(cudaStream_t st, const AsyncParams *params_dev, int grid, int block, const cudaAccessPolicyWindow *window)
{
   cudaLaunchConfig_t cfg = {};
   cfg.gridDim = dim3(grid);
   cfg.blockDim = dim3(block);
   cfg.dynamicSmemBytes = 0;
   cfg.stream = st;
   cudaLaunchAttribute attrs[2];
   int na = 0;
   attrs[na].id = cudaLaunchAttributeCooperative;
   attrs[na].val.cooperative = 1;
   na++;
   if (window && window->num_bytes > 0) {
      attrs[na].id = cudaLaunchAttributeAccessPolicyWindow;
      attrs[na].val.accessPolicyWindow = *window;
      na++;
   }
   cfg.attrs = attrs;
   cfg.numAttrs = na;
   const cudaError_t e = cudaLaunchKernelEx(&cfg, k_async_amg<false, true>, params_dev);
   return e == cudaSuccess ? 1 : -(int)e;
}

// ---- host side: the per-group programs (pure host code, no CUDA call) ------------------------------------------------
namespace {

struct ProgBuilder {
   const amgb_options &o;
   int L;
   bool symmetric, fact0;
   std::vector<AsyncOpSym> &ops;

   static AsyncOpSym blank(int type)
   {
      AsyncOpSym s;
      memset(&s, 0, sizeof(s));
      s.type = type;
      s.mat_kind = -1; s.mat_level = -1;
      s.x = s.y = s.b = s.c = s.rs = s.b2 = s.xs = s.red = s.red_copy = s.acc = AV_NONE;
      s.barrier = 1;
      s.red_scale = 1.0;
      return s;
   }
   int rs_id(int l) const { return o.smoother == AMGB_SMOOTH_L1_JACOBI ? AV_ID(AV_INVL1, l) : AV_ID(AV_WS, l); }
   AsyncOpSym &spmv(int kind, int level, int sval, int x, int y, double alpha, double beta, int b, double gamma = 0.0, int c = AV_NONE,
                    int rs = AV_NONE)
   {
      AsyncOpSym s = blank(AOP_SPMV);
      s.mat_kind = kind; s.mat_level = level; s.sval = sval; s.x = x; s.y = y; s.level = level;
      s.alpha = alpha; s.beta = beta; s.b = b; s.gamma = gamma; s.c = c; s.rs = rs;
      ops.push_back(s);
      return ops.back();
   }
   AsyncOpSym &vec(int type, int level, int x, int y)
   {
      AsyncOpSym s = blank(type);
      s.level = level; s.x = x; s.y = y;
      ops.push_back(s);
      return ops.back();
   }
   // e = S_l f from a zero guess (the dispatch of SMEM_Smooth, src/SMEM_Solve.cpp:264-323); returns the index of the op that
   // produces the final e (for epilogue fusion), or -1 when the result is produced by more than a single fused SpMV
   int smooth_zero(int l, int f, int e, int s1, int sweeps, bool sym)
   {
      const int sm = o.smoother;
      if (sm == AMGB_SMOOTH_ASYNC_GS || sm == AMGB_SMOOTH_SEMI_ASYNC_GS) {
         vec(AOP_ZERO, l, AV_NONE, e);
         if (sm == AMGB_SMOOTH_ASYNC_GS) { AsyncOpSym &g = vec(AOP_ASYNC_GS, l, f, e); g.sweeps = sweeps; }
         else for (int k = 0; k < sweeps; k++) { AsyncOpSym &g = vec(AOP_ASYNC_GS, l, f, e); g.sweeps = 1; }
         return -1;
      }
      if (sm == AMGB_SMOOTH_HYBRID_JGS) {
         { AsyncOpSym &g = vec(AOP_JGS, l, f, e); g.zero = 1; }
         for (int k = 1; k < sweeps; k++) {
            vec(AOP_COPY, l, e, s1);
            AsyncOpSym &g = vec(AOP_JGS, l, f, e);
            g.zero = 0; g.c = s1;                      // c = u_prev
         }
         return -1;
      }
      const int rs = rs_id(l);
      if (sym) {
         // sweep 1: e = rs o (2f - (A diag(rs)) f)      (src/SMEM_Smooth.cpp:655-695 in one pass)
         spmv(AMGB_MAT_A, l, 1, f, e, -1.0, 2.0, f, 0.0, AV_NONE, rs);
         for (int k = 1; k < sweeps; k++) {
            spmv(AMGB_MAT_A, l, 0, e, s1, -1.0, 1.0, f);
            spmv(AMGB_MAT_A, l, 1, s1, e, -1.0, 2.0, s1, 0.0, AV_NONE, rs);
         }
         return (int)ops.size() - 1;
      }
      // (L1-)Jacobi: u = rs o f, then u <- u + rs o (f - A u_prev), ping-pong so that the result lands in e
      int cur = ((sweeps - 1) & 1) ? s1 : e, oth = (cur == e) ? s1 : e;
      { AsyncOpSym &g = vec(AOP_SCALE, l, f, cur); g.rs = rs; }
      for (int k = 1; k < sweeps; k++) {
         spmv(AMGB_MAT_A, l, 0, cur, oth, -1.0, 1.0, f, 1.0, cur, rs);
         std::swap(cur, oth);
      }
      return sweeps == 1 ? (int)ops.size() - 1 : -1;
   }
};

}  // namespace

int async_build_program(const amgb_options &o, int L, bool symmetric, bool fact0, int q, std::vector<AsyncOpSym> &ops, bool partitioned)
{
   const bool multadd = o.solver == AMGB_SOLVER_ASYNC_MULTADD || o.solver == AMGB_SOLVER_MULTADD;
   const bool global = o.res_compute_type != 0, read_res = o.read_type != 0, semi = o.async_type != 0;
   const bool jac = o.smoother == AMGB_SMOOTH_JACOBI || o.smoother == AMGB_SMOOTH_L1_JACOBI;
   if (global && (!multadd || !jac || read_res || semi)) return AMGB_EINVAL;   // src/SMEM_Main.cpp:650-660: async Multadd only
   if (semi && read_res) return AMGB_EINVAL;
   if (fact0 && !(multadd && symmetric && jac)) return AMGB_EINVAL;
   ProgBuilder B{o, L, symmetric, fact0, ops};
   const int U = AV_ID(AV_U, 0), F = AV_ID(AV_F, 0), RS = AV_ID(AV_RS, 0), UL = AV_ID(AV_UL, 0), T0 = AV_ID(AV_T0, 0),
             FACC = AV_ID(AV_FACC, 0);
   auto Rv = [](int l) { return AV_ID(AV_R, l); };
   auto Ev = [](int l) { return AV_ID(AV_E, l); };
   auto Tv = [](int l) { return AV_ID(AV_T, l); };
   auto Wv = [](int l) { return AV_ID(AV_W, l); };
   // The coarsest level's correction is identically zero in the SMEM reference (direct solve commented out, :112-131): its
   // restrict / prolong / residual work adds exactly 0.0 to u, so this group only keeps the correction count and the
   // stop protocol.  With amgb_options.coarse_solve (DMEM's convention: AddCycle solves the coarsest grid directly,
   // src/DMEM_Add.cpp:262-264) it is a working group like the others: e_{L-1} = A_{L-1}^{-1} r_{L-1}.
   const bool direct = o.coarse_solve != 0 && L > 1;
   if (direct && global) return AMGB_EINVAL;
   const bool idle = (q == L - 1) && !direct;
   const bool coarse_q = direct && q == L - 1;
   const int rs0 = B.rs_id(0);
   if (global && !idle) {
      // all CTAs of the working groups: smooth level 0 on this CTA's rows, u += u_fine (:35-60).  The reference reads the group's copy of the shared
      // residual; here the shared residual itself (the copy only exists for the chain's sake, and the idle coarsest
      // group has none)
      if (symmetric) {
         AsyncOpSym &s = B.spmv(AMGB_MAT_A, 0, 1, RS, AV_NONE, -1.0, 2.0, RS, 0.0, AV_NONE, rs0);
         s.range = 1; s.red = U; s.barrier = 0;
      } else {
         AsyncOpSym &s = B.vec(AOP_SCALE, 0, RS, AV_NONE);
         s.rs = rs0; s.range = 1; s.red = U; s.barrier = 0;
      }
   }
   bool fused_update = false;
   if (!idle) {
      // ---- restriction chain (:93-108); level-0 transfers factorised: t_0 = r_0 - A_0 diag(w/d) r_0, r_1 = R_0 t_0
      const int coarsest = (multadd || coarse_q) ? q : q + 1;
      for (int l = 0; l < coarsest && l < L - 1; l++) {
         if (fact0 && l == 0) {
            B.spmv(AMGB_MAT_A, 0, 1, Rv(0), T0, -1.0, 1.0, Rv(0));
            B.spmv(AMGB_MAT_R, 0, 0, T0, Rv(1), 1.0, 0.0, AV_NONE);
         } else B.spmv(AMGB_MAT_R, l, 0, Rv(l), Rv(l + 1), 1.0, 0.0, AV_NONE);
      }
      // ---- correction on the group's level (:134-207)
      int last = -1;
      if (coarse_q) {
         B.spmv(AMAT_AINV, q, 0, Rv(q), Ev(q), 1.0, 0.0, AV_NONE);
         last = (int)ops.size() - 1;
      } else if (multadd) last = B.smooth_zero(q, Rv(q), Ev(q), Tv(q), o.num_fine_smooth_sweeps, symmetric);
      else {
         // AFACx (:153-206): u_c = S_{q+1} r_{q+1}; e = P u_c; r_f = r_q - A_q e; u_f = S_q r_f
         const int cl = q + 1;
         B.smooth_zero(cl, Rv(cl), Tv(cl), Wv(cl), o.num_coarse_smooth_sweeps, false);
         B.spmv(AMGB_MAT_P, q, 0, Tv(cl), Tv(q), 1.0, 0.0, AV_NONE);
         B.spmv(AMGB_MAT_A, q, 0, Tv(q), Wv(q), -1.0, 1.0, Rv(q));
         last = B.smooth_zero(q, Wv(q), Ev(q), Tv(q), o.num_fine_smooth_sweeps, false);
      }
      // ---- prolongation chain (:211-224); level 0 factorised: v = P_0 e_1, e_0 = v - (w/d) o (A_0 v)
      for (int l = q - 1; l >= 0; l--) {
         if (fact0 && l == 0) {
            // (row-partitioned solve: the prolongation side gets a scratch vector of its own -- a neighbour GPU that is half
            //  an iteration ahead or behind must never find the restriction side's t_0 in the ghost slots of v, or vice versa)
            const int V0 = partitioned ? Wv(0) : T0;
            B.spmv(AMGB_MAT_P, 0, 0, Ev(1), V0, 1.0, 0.0, AV_NONE);
            AsyncOpSym &s = B.spmv(AMGB_MAT_A, 0, 0, V0, Ev(0), -1.0, 0.0, AV_NONE, 0.0, AV_NONE, rs0);
            s.xs = V0; s.xself = 1.0;
         } else B.spmv(AMGB_MAT_P, l, 0, Ev(l + 1), Ev(l), 1.0, 0.0, AV_NONE);
         last = (int)ops.size() - 1;
      }
      // ---- the fine-level result e_0 is produced by ops[last] when that is a single SpMV / scale: fuse the update into it
      const bool can_fuse = last >= 0 && !semi && (ops[last].type == AOP_SPMV || (ops[last].type == AOP_SCALE && q == 0));
      if (read_res) {
         // -read_type res (:227-236,285-296): f_k += e_0; y = A_0 e_0; r -= y (shared, reduction); r_k = r
         if (last >= 0 && ops[last].type == AOP_SPMV) ops[last].acc = FACC;
         else { AsyncOpSym &a = B.vec(AOP_UPDATE, 0, Ev(0), AV_NONE); a.acc = FACC; }                    // (acc-only update)
         AsyncOpSym &s = B.spmv(AMGB_MAT_A, 0, 0, Ev(0), AV_NONE, 1.0, 0.0, AV_NONE);
         s.red = RS; s.red_scale = -1.0; s.red_copy = Rv(0);
         fused_update = true;
      } else if (can_fuse) {
         AsyncOpSym &s = ops[last];
         s.red = U;
         if (!global) s.red_copy = UL;
         if (s.type == AOP_SPMV) s.y = AV_NONE;       // e_0 itself is not needed any more
         fused_update = true;
      }
      if (!fused_update) {
         // ---- u += e (atomic), private copy (:285-301); SEMI_ASYNC: one critical section per group (:238-283)
         if (semi) { AsyncOpSym &l = B.vec(AOP_LOCK, 0, AV_NONE, AV_NONE); (void)l; }
         AsyncOpSym &u = B.vec(AOP_UPDATE, 0, Ev(0), AV_NONE);
         u.red = U; u.red_copy = global ? AV_NONE : UL; u.locked = semi ? 1 : 0;
         if (semi) B.vec(AOP_UNLOCK, 0, AV_NONE, AV_NONE).barrier = 0;
         else u.barrier = 0;                           // (the count / stop operation starts with a barrier of its own)
      }
   }
   B.vec(AOP_COUNT_STOP, 0, AV_NONE, AV_NONE).barrier = 0;
   if (global && !idle) {
      // ---- all working CTAs: residual of this CTA's rows from the shared u into the shared r, then the group's copy (:356-416)
      AsyncOpSym &s = B.spmv(AMGB_MAT_A, 0, 0, U, RS, -1.0, 1.0, F);
      s.range = 1;
      B.vec(AOP_COPY, 0, RS, Rv(0));
   } else if (!idle && !read_res) {
      // ---- private residual from the private copy (:338-351)
      B.spmv(AMGB_MAT_A, 0, 0, UL, Rv(0), -1.0, 1.0, F);
   }
   return AMGB_OK;
}

// The program of group q of the asynchronous implicit extended-system solver (SMEM_ExtendedSystemSolve with
// IMPLICIT_EXTENDED_SYSTEM_BPX and async_flag = 1, src/SMEM_ExtendedSystem.cpp:305,365,474-479,636-652): the reference's thread
// group of level q rebuilds both chains it needs from whatever the other groups have written so far --
//   z1_{L-1} = u_{L-1},  z1_j = P_j z1_{j+1} + u_j  (j = L-2 .. q);   z2_0 = 0,  z2_{j+1} = R_j (z2_j + e_j)  (j = 0 .. q-1)
//   r_q = f_q - z2_q - A_q z1_q;  u_q <- y_q + omega (delta rs o r_q + u_q - y_q), y_q <- old u_q;  e_q = A_q u_q;  count / stop
// It writes u_q, y_q, e_q and its own chain vectors only; it reads u_j (j >= q) and e_j (j < q).
int async_build_ext_program(const amgb_options &o, int L, int q, std::vector<AsyncOpSym> &ops)
{
   if (o.smoother != AMGB_SMOOTH_JACOBI && o.smoother != AMGB_SMOOTH_L1_JACOBI) return AMGB_EINVAL;
   if (L < 1 || L > AMGB_MAX_LEVELS || q < 0 || q >= L) return AMGB_EINVAL;
   ProgBuilder B{o, L, true, false, ops};
   // ---- prolongation chain; the last one needs no barrier of its own when the restriction chain follows (it does not read z1)
   int z1 = AV_ID(AV_XU, L - 1);
   for (int j = L - 2; j >= q; j--) {
      B.spmv(AMGB_MAT_P, j, 0, z1, AV_ID(AV_XZ1, j), 1.0, 1.0, AV_ID(AV_XU, j)).barrier = (j == q && q > 0) ? 0 : 1;
      z1 = AV_ID(AV_XZ1, j);
   }
   // ---- restriction chain: on the levels it passes, the SpMV's epilogue adds e_{j+1} (z2_{j+1} alone is never read there)
   int z2 = AV_ID(AV_XE, 0);
   for (int j = 0; j < q; j++) {
      const bool last = j + 1 == q;
      B.spmv(AMGB_MAT_R, j, 0, z2, AV_ID(AV_XZ2, j + 1), 1.0, last ? 0.0 : 1.0, last ? AV_NONE : AV_ID(AV_XE, j + 1));
      z2 = AV_ID(AV_XZ2, j + 1);
   }
   // ---- residual and its sum of squares, Chebyshev update, e_q (no group reads e_{L-1})
   {
      AsyncOpSym &r = B.spmv(AMGB_MAT_A, q, 0, z1, AV_ID(AV_XR, q), -1.0, 1.0, AV_ID(AV_XF, q));
      r.type = AOP_EXT_RESID;
      if (q > 0) { r.b2 = z2; r.beta2 = -1.0; }
   }
   {
      AsyncOpSym &c = B.vec(AOP_EXT_CHEBY, q, AV_ID(AV_XR, q), AV_ID(AV_XU, q));
      c.c = AV_ID(AV_XY, q);
      c.rs = B.rs_id(q);
   }
   if (q < L - 1) B.spmv(AMGB_MAT_A, q, 0, AV_ID(AV_XU, q), AV_ID(AV_XE, q), 1.0, 0.0, AV_NONE);
   B.vec(AOP_EXT_STOP, q, AV_NONE, AV_NONE).barrier = 0;      // (it ends with the group's decision, a barrier of its own)
   return AMGB_OK;
}

// ---- host side: build the parameter block once, run ---------------------------------------------
static bool async_heavy(const amgb_options &o)
{
   return o.smoother == AMGB_SMOOTH_HYBRID_JGS || o.smoother == AMGB_SMOOTH_ASYNC_GS || o.smoother == AMGB_SMOOTH_SEMI_ASYNC_GS;
}

// estimated seconds-equivalent cost of streaming one operator once (bytes over the fraction of the HBM roofline its storage
// reaches in the stand-alone kernels, profiles/README.md): only the RATIOS matter, they seed the CTA-group sizes
double async_op_cost(const DevCSR &M, long sell_entries)
{
   if (M.su_desc) return (32.0 * M.nrows) / 0.8;
   if (M.sell_slices > 0) return (12.0 * (double)sell_entries + 16.0 * M.nrows) / (M.sell_perm ? 0.55 : 0.85);
   return (12.0 * M.nnz + 16.0 * M.nrows) / 0.4;
}

static int async_prepare(amgb_ctx *c)
{
   if (c->async_ready) return AMGB_OK;
   const int L = c->L;
   const amgb_options &o = c->opt;
   const bool multadd = o.solver == AMGB_SOLVER_ASYNC_MULTADD || o.solver == AMGB_SOLVER_MULTADD;
   const bool jac = o.smoother == AMGB_SMOOTH_JACOBI || o.smoother == AMGB_SMOOTH_L1_JACOBI;
   // factorised level-0 transfers: plain P_0 / R_0 were uploaded (amgb_options.factor_level0)
   const bool fact0 = o.factor_level0 && multadd && c->symmetric && jac && L >= 2;
   const bool global = o.res_compute_type != 0, read_res = o.read_type != 0;
   const bool heavy = async_heavy(o);
   const int first = global ? 1 : 0;
   if (global && L < 2) return amgb_fail(c, AMGB_EINVAL, "-res_compute_type global needs at least two levels");
   AsyncParams hp;
   memset(&hp, 0, sizeof(hp));
   hp.num_levels = L;
   hp.first_group = first;
   hp.smoother = o.smoother;
   hp.jgs_block_rows = o.jgs_block_rows;
   hp.n0 = c->A[0].nrows;
   for (int l = 0; l < L; l++) {
      const double avg = c->A[l].nrows > 0 ? (double)c->A[l].nnz / c->A[l].nrows : 0.0;
      hp.jgs_lpb[l] = o.jgs_block_rows > AMGB_JGS_BMAX ? 0 : (avg <= 5.0 ? 4 : (avg <= 10.0 ? 8 : (avg <= 20.0 ? 16 : 32)));
      hp.A[l] = c->A[l];
      if (l < L - 1) { hp.P[l] = c->P[l]; hp.R[l] = c->R[l]; }
   }
   hp.Ainv = c->Ainv;
   int rc;
   // ---- programs (symbolic), then the vectors they name
   std::vector<AsyncOpSym> sym;
   std::vector<int> op_begin(L + 1, 0);
   for (int q = 0; q < L; q++) {
      op_begin[q] = (int)sym.size();
      if (q >= first && (rc = async_build_program(o, L, c->symmetric, fact0, q, sym)))
         return amgb_fail(c, rc, "this combination of asynchronous options is not implemented (see amgb_options)");
   }
   op_begin[L] = (int)sym.size();
   const int n0 = c->A[0].nrows;
   double *r_shared = nullptr;
   if (global || read_res) {
      if ((rc = amgb_dev_alloc_bytes(c, (void **)&r_shared, sizeof(double) * (size_t)n0, true))) return rc;
   }
   c->async_r_shared = r_shared;
   c->async_vec.assign((size_t)L * 12 * 64, nullptr);        // [group][kind][level] -> device pointer (group-private kinds)
   auto slot = [&](int q, int id) -> double *& { return c->async_vec[((size_t)q * 12 + (size_t)(id / 64)) * 64 + (size_t)(id % 64)]; };
   auto resolve = [&](int q, int id, double **out) -> int {
      *out = nullptr;
      if (id == AV_NONE) return AMGB_OK;
      const int kind = id / 64, l = id % 64;
      switch (kind) {
         case AV_F: *out = c->f; return AMGB_OK;
         case AV_U: *out = c->u; return AMGB_OK;
         case AV_RS: *out = r_shared; return AMGB_OK;
         case AV_WS: *out = c->ws[l]; return AMGB_OK;
         case AV_INVL1: *out = c->inv_l1[l]; return AMGB_OK;
         default: break;
      }
      double *&p = slot(q, id);
      if (!p) {
         const int lv = (kind == AV_UL || kind == AV_T0 || kind == AV_FACC) ? 0 : l;
         int r2 = amgb_dev_alloc_bytes(c, (void **)&p, sizeof(double) * (size_t)c->A[lv].nrows, true);
         if (r2) return r2;
      }
      *out = p;
      return AMGB_OK;
   };
   std::vector<AsyncOp> dev_ops(sym.size());
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
         if ((rc = resolve(q, s.xs, &t))) return rc; d.e.xs = t;
         if ((rc = resolve(q, s.red, &t))) return rc; d.e.red = t;
         if ((rc = resolve(q, s.red_copy, &t))) return rc; d.e.red_copy = t;
         if ((rc = resolve(q, s.acc, &t))) return rc; d.e.acc = t;
      }
   // every working group starts from a copy of r0 and of u (src/SMEM_Async_AMG.cpp:10-15): make sure those vectors exist
   for (int q = first; q < L; q++) {
      double *t;
      if ((rc = resolve(q, AV_ID(AV_R, 0), &t))) return rc;
      if (!global && !read_res && (rc = resolve(q, AV_ID(AV_UL, 0), &t))) return rc;
   }
   AsyncOp *d_ops = nullptr;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&d_ops, sizeof(AsyncOp) * std::max<size_t>(dev_ops.size(), 1), false))) return rc;
   CUDA_OK(c, cudaMemcpyAsync(d_ops, dev_ops.data(), sizeof(AsyncOp) * dev_ops.size(), cudaMemcpyHostToDevice, c->stream));
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   hp.ops = d_ops;
   for (int q = 0; q <= L; q++) hp.op_begin[q] = op_begin[q];
   // ---- CTA groups: seeded by a cost model of every group's program, refined from measured group times at the first solve
   std::vector<double> work(L, 0.0);
   for (int q = first; q < L; q++) {
      double w = 0.0;
      for (int i = op_begin[q]; i < op_begin[q + 1]; i++) {
         const AsyncOpSym &s = sym[i];
         if (s.range) continue;                       // CTA-slice work is the same for every CTA
         if (s.type == AOP_SPMV) {
            const DevCSR &M = s.mat_kind == AMGB_MAT_A ? c->A[s.mat_level] : (s.mat_kind == AMGB_MAT_P ? c->P[s.mat_level] : (s.mat_kind == AMGB_MAT_R ? c->R[s.mat_level] : c->Ainv));
            auto it = c->sell_entries.find(&M);
            w += async_op_cost(M, it == c->sell_entries.end() ? 0 : it->second) + 24.0 * M.nrows;
         } else if (s.type == AOP_JGS || s.type == AOP_ASYNC_GS) {
            w += 4.0 * 12.0 * c->A[s.level].nnz * std::max(1, s.sweeps);
         } else if (s.type != AOP_COUNT_STOP && s.type != AOP_LOCK && s.type != AOP_UNLOCK) {
            w += 24.0 * c->A[s.level].nrows;
         }
      }
      work[q] = w;
   }
   c->async_work = work;
   c->async_heavy = heavy;
   c->async_first = first;
   int grid = async_max_grid(kABlock, heavy);
   grid = std::max(L - first, std::min(grid, n0 / 64 + L));      // small problems: no more CTAs than there is work for
   if (grid < L - first) return amgb_fail(c, AMGB_ECUDA, "cooperative grid %d smaller than the number of level groups %d", grid, L - first);
   c->async_grid = grid;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&hp.barrier_count, sizeof(unsigned int) * AMGB_MAX_LEVELS, true))) return rc;
   unsigned int *gen;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&gen, sizeof(unsigned int) * AMGB_MAX_LEVELS, true))) return rc;
   hp.barrier_gen = gen;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&hp.num_correct, sizeof(int) * AMGB_MAX_LEVELS, true))) return rc;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&hp.group_stop, sizeof(int) * AMGB_MAX_LEVELS, true))) return rc;
   int *flag;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&flag, sizeof(int) * 4, true))) return rc;
   hp.converge_flag = flag;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&hp.lock, sizeof(int) * 4, true))) return rc;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&hp.group_ns, sizeof(unsigned long long) * AMGB_MAX_LEVELS, true))) return rc;
   hp.u = c->u;
   if (o.l2_persist && c->arena_used > 0) {
      // pin the coarse hierarchy in L2 for the persistent kernel (launch attribute, see launch_async)
      c->window.base_ptr = c->arena;
      c->window.num_bytes = std::min(c->arena_used, c->max_window);
      c->window.hitRatio = 1.0f;
      c->window.hitProp = cudaAccessPropertyPersisting;
      c->window.missProp = cudaAccessPropertyStreaming;
      c->window_valid = true;
   }
   c->async_host = new AsyncParams(hp);
   if ((rc = amgb_dev_alloc_bytes(c, &c->async_params_dev, sizeof(AsyncParams), false))) return rc;
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   c->async_ready = true;
   return AMGB_OK;
}

// CTA groups proportional to `work` (one CTA per group at least; a group whose work is zero -- the idle coarsest group --
// keeps exactly one): largest-remainder distribution
void async_assign_groups(amgb_ctx *c, const std::vector<double> &work)
{
   AsyncParams &hp = *c->async_host;
   const int L = c->L, first = c->async_first, grid = c->async_grid;
   async_deal_ctas(work, L, first, grid, hp.cta_begin);
   hp.slice_ctas = std::max(1, L > 1 ? hp.cta_begin[L - 1] : hp.cta_begin[L]);      // CTAs of the working groups
   c->async_cta_begin.assign(hp.cta_begin, hp.cta_begin + L + 1);
   c->async_grid_used = hp.cta_begin[L];
}

void async_deal_ctas(const std::vector<double> &work, int L, int first, int grid, int *cta_begin)
{
   double tot = 0.0;
   for (int q = first; q < L; q++) tot += work[q];
   std::vector<int> ctas(L, 0);
   int left = grid;
   for (int q = first; q < L; q++) { ctas[q] = 1; left--; }
   if (tot > 0.0) {
      std::vector<double> want(L, 0.0);
      for (int q = first; q < L; q++) want[q] = work[q] / tot * grid;
      for (int q = first; q < L; q++) {
         int extra = (int)std::floor(std::max(0.0, want[q] - 1.0));
         extra = std::min(extra, left);
         ctas[q] += extra;
         left -= extra;
      }
      // the remainder goes to the groups furthest below their share
      while (left > 0) {
         int best = -1;
         double gap = -1e300;
         for (int q = first; q < L; q++) {
            if (work[q] <= 0.0) continue;
            const double g = want[q] - ctas[q];
            if (g > gap) { gap = g; best = q; }
         }
         if (best < 0) break;
         ctas[best]++; left--;
      }
   }
   for (int q = 0; q <= first; q++) cta_begin[q] = 0;
   for (int q = first; q < L; q++) cta_begin[q + 1] = cta_begin[q] + ctas[q];
}

void amgb_async_teardown(amgb_ctx *c)
{
   delete c->async_host;
   c->async_host = nullptr;
}

// one launch of the persistent kernel from the resident f, u; r0 and ||r0|| first (src/SMEM_Solve.cpp:60-70)
static int async_run(amgb_ctx *c, int num_cycles, int converge_type, double *r0_out, double *solve_seconds)
{
   AsyncParams &hp = *c->async_host;
   const int L = c->L, n0 = c->A[0].nrows, first = c->async_first;
   const bool global = c->opt.res_compute_type != 0, read_res = c->opt.read_type != 0;
   int rc;
   hp.num_cycles = num_cycles;
   hp.converge_type = converge_type;
   enq_residual(c);
   double ss;
   if ((rc = amgb_fetch_scalar(c, &ss))) return rc;
   if (r0_out) *r0_out = sqrt(ss);
   auto vec = [&](int q, int kind) { return c->async_vec[((size_t)q * 12 + (size_t)kind) * 64]; };
   // every group starts from a copy of r0 (src/SMEM_Async_AMG.cpp:10-15) and of u
   for (int q = first; q < L; q++) {
      if (double *r = vec(q, AV_R)) CUDA_OK(c, cudaMemcpyAsync(r, c->r[0], sizeof(double) * n0, cudaMemcpyDeviceToDevice, c->stream));
      if (double *ul = vec(q, AV_UL)) CUDA_OK(c, cudaMemcpyAsync(ul, c->u, sizeof(double) * n0, cudaMemcpyDeviceToDevice, c->stream));
      if (double *fa = vec(q, AV_FACC)) CUDA_OK(c, cudaMemsetAsync(fa, 0, sizeof(double) * n0, c->stream));
   }
   if (global || read_res) CUDA_OK(c, cudaMemcpyAsync(c->async_r_shared, c->r[0], sizeof(double) * n0, cudaMemcpyDeviceToDevice, c->stream));
   CUDA_OK(c, cudaMemsetAsync(hp.barrier_count, 0, sizeof(unsigned int) * AMGB_MAX_LEVELS, c->stream));
   CUDA_OK(c, cudaMemsetAsync((void *)hp.barrier_gen, 0, sizeof(unsigned int) * AMGB_MAX_LEVELS, c->stream));
   CUDA_OK(c, cudaMemsetAsync(hp.num_correct, 0, sizeof(int) * AMGB_MAX_LEVELS, c->stream));
   CUDA_OK(c, cudaMemsetAsync(hp.group_stop, 0, sizeof(int) * AMGB_MAX_LEVELS, c->stream));
   CUDA_OK(c, cudaMemsetAsync((void *)hp.converge_flag, 0, sizeof(int) * 4, c->stream));
   CUDA_OK(c, cudaMemsetAsync(hp.lock, 0, sizeof(int) * 4, c->stream));
   CUDA_OK(c, cudaMemsetAsync(hp.group_ns, 0, sizeof(unsigned long long) * AMGB_MAX_LEVELS, c->stream));
   CUDA_OK(c, cudaMemcpyAsync(c->async_params_dev, &hp, sizeof(AsyncParams), cudaMemcpyHostToDevice, c->stream));
   CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
   const int lr = launch_async(c->stream, (const AsyncParams *)c->async_params_dev, c->async_grid_used, kABlock, c->async_heavy,
                               c->window_valid ? &c->window : nullptr);
   if (lr < 0) return amgb_fail(c, AMGB_ECUDA, "cooperative launch failed: %s", cudaGetErrorString((cudaError_t)(-lr)));
   c->launches += 1;
   CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
   CUDA_OK(c, cudaEventSynchronize(c->ev1));
   float ms = 0;
   cudaEventElapsedTime(&ms, c->ev0, c->ev1);
   if (solve_seconds) *solve_seconds = ms * 1e-3;
   if (read_res) {
      // u += sum over the levels of their accumulated corrections, level after level (:416-426)
      for (int q = first; q < L; q++)
         if (double *fa = vec(q, AV_FACC)) c->launches += launch_add(c->cfg, c->stream, n0, fa, c->u);
   }
   CUDA_OK(c, cudaGetLastError());
   return AMGB_OK;
}

extern "C" int amgb_solve_async(amgb_ctx *c, int num_cycles, int converge_type, int *corrections, double *relres,
                                double *solve_seconds)
{
   NEED_READY(c);
   if (num_cycles < 1) return amgb_fail(c, AMGB_EINVAL, "num_cycles < 1");
   if (c->opt.coarse_solve && c->L > 1 && !c->Ainv.rp) return amgb_fail(c, AMGB_ESTATE, "coarse_solve: the inverse of the coarsest operator was not built");
   for (int *b : c->jgs_bounds)
      if (b) return amgb_fail(c, AMGB_EINVAL, "explicit hybrid-JGS block lists are implemented for the synchronous cycles");
   int rc;
   if ((rc = async_prepare(c))) return rc;
   AsyncParams &hp = *c->async_host;
   const int L = c->L, n0 = c->A[0].nrows;
   if (!c->async_balanced) {
      // CTA-group balancing: a LOCAL-rule solve lasts as long as its slowest group, so the groups are sized from MEASURED
      // time -- two short launches on a scratch copy of u (restored afterwards), each followed by a re-deal of the CTAs
      // in proportion to (CTAs x time) of every group.  The reference sizes its thread groups from a static work model
      // (src/SMEM_Setup.cpp:770-868,1083-1160); that model seeds the first launch here.
      async_assign_groups(c, c->async_work);
      const char *env = getenv("AMGB_ASYNC_BALANCE");
      const int rounds = env ? atoi(env) : 2;
      if (rounds > 0 && L - c->async_first > 2) {
         CUDA_OK(c, cudaMemcpyAsync(c->u_outer, c->u, sizeof(double) * n0, cudaMemcpyDeviceToDevice, c->stream));
         for (int it = 0; it < rounds; it++) {
            if ((rc = async_run(c, 3, AMGB_CONVERGE_LOCAL, nullptr, nullptr))) return rc;
            std::vector<unsigned long long> ns(AMGB_MAX_LEVELS);
            CUDA_OK(c, cudaMemcpy(ns.data(), hp.group_ns, sizeof(unsigned long long) * AMGB_MAX_LEVELS, cudaMemcpyDeviceToHost));
            std::vector<double> work(L, 0.0);
            for (int q = c->async_first; q < L; q++) {
               const int nct = hp.cta_begin[q + 1] - hp.cta_begin[q];
               work[q] = c->async_work[q] > 0.0 ? (double)nct * (double)ns[q] : 0.0;
            }
            async_assign_groups(c, work);
            CUDA_OK(c, cudaMemcpyAsync(c->u, c->u_outer, sizeof(double) * n0, cudaMemcpyDeviceToDevice, c->stream));
         }
      }
      c->async_balanced = true;
   }
   double r0 = 0.0;
   if ((rc = async_run(c, num_cycles, converge_type, &r0, solve_seconds))) return rc;
   // final residual on the shared u (src/SMEM_Solve.cpp:82-91)
   enq_residual(c);
   double ss;
   if ((rc = amgb_fetch_scalar(c, &ss))) return rc;
   if (relres) *relres = sqrt(ss) / r0;
   if (corrections) {
      std::vector<int> h(AMGB_MAX_LEVELS);
      CUDA_OK(c, cudaMemcpy(h.data(), hp.num_correct, sizeof(int) * AMGB_MAX_LEVELS, cudaMemcpyDeviceToHost));
      for (int l = 0; l < L; l++) corrections[l] = h[l];
   }
   CUDA_OK(c, cudaGetLastError());
   return AMGB_OK;
}

extern "C" int amgb_async_groups(amgb_ctx *c, int *cta_begin /* num_levels+1 */, int *grid)
{
   NEED_READY(c);
   int rc;
   if ((rc = async_prepare(c))) return rc;
   if (c->async_cta_begin.empty()) async_assign_groups(c, c->async_work);
   for (int l = 0; l <= c->L; l++) cta_begin[l] = c->async_cta_begin[l];
   if (grid) *grid = c->async_grid_used;
   return AMGB_OK;
}

// nanoseconds every level group spent inside the last launch of the persistent kernel (group root's %globaltimer)
extern "C" int amgb_async_group_times(amgb_ctx *c, double *seconds /* num_levels */)
{
   NEED_READY(c);
   if (!c->async_ready || !seconds) return amgb_fail(c, AMGB_ESTATE, "no asynchronous solve yet");
   std::vector<unsigned long long> ns(AMGB_MAX_LEVELS);
   CUDA_OK(c, cudaMemcpy(ns.data(), c->async_host->group_ns, sizeof(unsigned long long) * AMGB_MAX_LEVELS, cudaMemcpyDeviceToHost));
   for (int l = 0; l < c->L; l++) seconds[l] = 1e-9 * (double)ns[l];
   return AMGB_OK;
}

// Host-only probe for the CPU test suite: the programs the persistent kernel would interpret for these options and this
// number of levels (no CUDA call).  ops: caller's array of max_ops AsyncOpSym; op_begin[num_levels + 1].
extern "C" int amgb_async_program(const amgb_options *o, int num_levels, int symmetric, int fact0, void *ops, int max_ops, int *op_begin)
{
   if (!o || !ops || !op_begin || num_levels < 1 || num_levels > AMGB_MAX_LEVELS) return AMGB_EINVAL;
   std::vector<AsyncOpSym> sym;
   const int first = o->res_compute_type != 0 ? 1 : 0;
   for (int q = 0; q < num_levels; q++) {
      op_begin[q] = (int)sym.size();
      if (q < first) continue;
      int rc = async_build_program(*o, num_levels, symmetric != 0, fact0 != 0, q, sym);
      if (rc) return rc;
   }
   op_begin[num_levels] = (int)sym.size();
   if ((int)sym.size() > max_ops) return AMGB_ENOMEM;
   memcpy(ops, sym.data(), sizeof(AsyncOpSym) * sym.size());
   return AMGB_OK;
}

// Host-only probe: the programs of amgb_solve_extended_implicit_async for these options and this number of levels.
extern "C" int amgb_ext_async_program(const amgb_options *o, int num_levels, void *ops, int max_ops, int *op_begin)
{
   if (!o || !ops || !op_begin || num_levels < 1 || num_levels > AMGB_MAX_LEVELS) return AMGB_EINVAL;
   std::vector<AsyncOpSym> sym;
   for (int q = 0; q < num_levels; q++) {
      op_begin[q] = (int)sym.size();
      const int rc = async_build_ext_program(*o, num_levels, q, sym);
      if (rc) return rc;
   }
   op_begin[num_levels] = (int)sym.size();
   if ((int)sym.size() > max_ops) return AMGB_ENOMEM;
   memcpy(ops, sym.data(), sizeof(AsyncOpSym) * sym.size());
   return AMGB_OK;
}

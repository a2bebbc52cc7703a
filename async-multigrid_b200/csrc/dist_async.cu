// dist_async.cu -- the asynchronous additive solve ROW-PARTITIONED over the GPUs of one box.
//
// Replaces DMEM_Add's asynchronous loop (src/DMEM_Add.cpp:101-130) with its correction / residual exchange
// (DMEM_AddCorrect_LocalRes / DMEM_AddResidual_LocalRes, src/DMEM_Add.cpp:391-556) and DMEM_Comm's Isend / Test engine
// (src/DMEM_Comm.cpp:81-382, :267-330).  The reference gives every GRID a group of MPI ranks; a rank holds a row range of its
// grid's operators, restricts / smooths / prolongs its piece of its grid's correction with hypre ParCSR matvecs inside the
// group, and ships fine-level corrections to the other grids with non-blocking messages that are consumed whenever they
// have arrived.  Here the partition is the synchronous path's (dist.cu: every level's rows in contiguous z-slab ranges, one
// range per GPU, small coarse levels replicated) and the asynchrony is the persistent kernel's (async.cu): every GPU runs
// ONE cooperative kernel whose CTA groups own the levels and loop over the SAME programs as on one GPU, on the GPU's row
// blocks; a group's vectors live in the extended layout [ghost_lo | owned | ghost_hi] and after every operation whose
// result a later SpMV of the group reads with ghosts, the group stores its boundary entries straight into the ghost slots
// of the same group's vector on the neighbour GPUs (AOP_PUSH: plain stores through CUDA-IPC peer mappings over NVLink).
// Entering a replicated level, every GPU stores its slice of the restricted residual into every peer's copy.  NOBODY WAITS:
// a group reads whatever its ghost slots hold -- the neighbour's values of this iteration or of the one before -- which is
// the reference's "use what has arrived" rule applied to every vector of the chain (all of them tend to zero with the
// residual; the multi-rank interpreter of the CPU suite, tests/dist_async_emulator.py, runs the same plans under random
// interleavings).  The shared u of a GPU's rows is updated only by that GPU's groups (fp64 reductions in its own memory);
// every group pushes the boundary of its private copy of u for its neighbours' residuals.  Stop rule: LOCAL -- every
// group on every GPU stops after num_cycles own corrections (src/DMEM_Add.cpp:119-127 with -converge_test_type local).
//
// Planning (dist_async_plan) is pure host code: the CPU suite interprets its output for 2 and 3 ranks and checks it, in the
// lock-step interleaving, against the single-GPU programs on the unpartitioned hierarchy.
#include "dist.h"
#include "async_team.cuh"
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <vector>
#include <omp.h>

// ---- host planning ----------------------------------------------------------------------------------------------------
namespace {

inline int vec_level(int id)
{
   const int kind = id / 64;
   return (kind == AV_UL || kind == AV_T0 || kind == AV_FACC || kind == AV_U || kind == AV_F || kind == AV_RS) ? 0 : id % 64;
}

inline int sym_role(const AsyncOpSym &s, int role)
{
   switch (role) {
      case DROLE_X: return s.x;
      case DROLE_Y: return s.y;
      case DROLE_B: return s.b;
      case DROLE_C: return s.c;
      case DROLE_RS: return s.rs;
      case DROLE_B2: return s.b2;
      case DROLE_XS: return s.xs;
      case DROLE_RED: return s.red;
      case DROLE_RED_COPY: return s.red_copy;
      default: return s.acc;
   }
}

}  // namespace

int dist_async_plan(const amgb_options &o, int L, int nranks, int rank, const DistLay *lay, bool symmetric, bool fact0, DistAsyncPlan &out)
{
   if (L < 1 || L > AMGB_MAX_LEVELS || nranks < 1 || rank < 0 || rank >= nranks || !lay) return AMGB_EINVAL;
   const bool multadd = o.solver == AMGB_SOLVER_ASYNC_MULTADD || o.solver == AMGB_SOLVER_MULTADD;
   const bool afacx = o.solver == AMGB_SOLVER_ASYNC_AFACX || o.solver == AMGB_SOLVER_AFACX;
   if (!multadd && !afacx) return AMGB_EINVAL;
   if (o.smoother != AMGB_SMOOTH_JACOBI && o.smoother != AMGB_SMOOTH_L1_JACOBI) return AMGB_EINVAL;
   if (o.res_compute_type || o.read_type || o.async_type) return AMGB_EINVAL;      // the shared-residual variants need a shared r
   if (o.coarse_solve && L > 1 && lay[(size_t)rank * L + (L - 1)].distributed) return AMGB_EINVAL;   // the direct coarse solve needs the coarsest level whole
   auto LAY = [&](int p, int l) -> const DistLay & { return lay[(size_t)p * L + l]; };
   int num_dist = 0;
   while (num_dist < L && LAY(rank, num_dist).distributed) num_dist++;
   for (int p = 0; p < nranks; p++)
      for (int l = 0; l < L; l++) {
         const DistLay &a = LAY(p, l);
         if ((a.distributed != 0) != (l < num_dist)) return AMGB_EINVAL;
         if (a.distributed) {
            if (p > 0 && a.send_lo != LAY(p - 1, l).halo_hi) return AMGB_EINVAL;
            if (p < nranks - 1 && a.send_hi != LAY(p + 1, l).halo_lo) return AMGB_EINVAL;
            if ((p == 0 && a.halo_lo) || (p == nranks - 1 && a.halo_hi)) return AMGB_EINVAL;
         }
      }
   out.ops.clear(); out.op_begin.assign(L + 1, 0); out.slot_off.assign(1, 0); out.slot_group.clear(); out.slot_vec.clear();
   std::map<std::pair<int, int>, int> slot_of;      // (group, vector id) -> slot
   auto slot = [&](int q, int id) -> int {
      auto key = std::make_pair(q, id);
      auto it = slot_of.find(key);
      if (it != slot_of.end()) return it->second;
      const int l = vec_level(id);
      long long len = 0;
      for (int p = 0; p < nranks; p++) {
         const DistLay &a = LAY(p, l);
         len = std::max(len, (long long)(a.distributed ? a.halo_lo + a.n_owned + a.halo_hi : a.n_global));
      }
      len = (len + 31) / 32 * 32 + 32;          // 256-byte granular, with slack for the kernels' 16-byte bulk reads
      const int s = (int)out.slot_group.size();
      out.slot_group.push_back(q); out.slot_vec.push_back(id);
      out.slot_off.push_back(out.slot_off.back() + len);
      slot_of[key] = s;
      return s;
   };
   auto off = [&](int p, int l) { const DistLay &a = LAY(p, l); return (long long)(a.distributed ? a.halo_lo : 0); };
   std::vector<AsyncOpSym> sym;
   for (int q = 0; q < L; q++) {
      out.op_begin[q] = (int)out.ops.size();
      sym.clear();
      int rc = async_build_program(o, L, symmetric, fact0, q, sym, true);
      if (rc) return rc;
      // vectors a later (or, the program being a loop, an earlier) SpMV of this group reads as its input
      auto read_by_spmv = [&](int id) {
         for (const AsyncOpSym &t : sym)
            if (t.type == AOP_SPMV && t.x == id) return true;
         return false;
      };
      for (size_t i = 0; i < sym.size(); i++) {
         const AsyncOpSym &s = sym[i];
         if (s.type == AOP_JGS || s.type == AOP_ASYNC_GS || s.type == AOP_LOCK || s.type == AOP_UNLOCK || s.range) return AMGB_EINVAL;
         DistAsyncOp d;
         memset(&d, 0, sizeof(d));
         d.type = s.type; d.mat_kind = s.mat_kind; d.mat_level = s.mat_level; d.sval = s.sval; d.barrier = s.barrier; d.level = s.level;
         d.alpha = s.alpha; d.beta = s.beta; d.gamma = s.gamma; d.beta2 = s.beta2; d.xself = s.xself; d.red_scale = s.red_scale;
         d.dst_rank = -1;
         // the restriction that enters the replicated tail writes this rank's slice of the (full-length) coarse residual
         const bool gather = s.type == AOP_SPMV && s.mat_kind == AMGB_MAT_R && num_dist > 0 && s.mat_level == num_dist - 1 && num_dist < L;
         for (int role = 0; role < DROLE_N; role++) {
            const int id = sym_role(s, role);
            d.slot[role] = DEXT_NONE; d.elem[role] = 0;
            if (id == AV_NONE) continue;
            const int kind = id / 64, l = vec_level(id);
            const bool whole = s.type == AOP_SPMV && role == DROLE_X;      // an SpMV input is addressed in the extended numbering
            long long e = whole ? 0 : off(rank, l);
            if (gather && role == DROLE_Y) e = LAY(rank, l).row_start;
            if (kind == AV_F) { d.slot[role] = DEXT_F; d.elem[role] = 0; continue; }
            if (kind == AV_U) { d.slot[role] = DEXT_U; d.elem[role] = e; continue; }
            if (kind == AV_WS || kind == AV_INVL1) { d.slot[role] = DEXT_WS0 - l; d.elem[role] = e; continue; }
            if (kind == AV_RS) return AMGB_EINVAL;
            d.slot[role] = slot(q, id);
            d.elem[role] = e;
         }
         // vectors this operation writes whose ghosts (or peers' copies) somebody reads
         int written[2] = {s.y, s.red_copy};
         bool pushes = false;
         for (int w = 0; w < 2; w++) {
            const int id = written[w];
            if (id == AV_NONE || id / 64 == AV_U) continue;
            const int l = vec_level(id);
            if ((l < num_dist && read_by_spmv(id)) || (w == 0 && gather)) pushes = true;
         }
         if (pushes) d.barrier = 1;       // the whole group's rows must be in place before their boundary leaves
         out.ops.push_back(d);
         for (int w = 0; w < 2; w++) {
            const int id = written[w];
            if (id == AV_NONE || id / 64 == AV_U) continue;
            const int l = vec_level(id);
            const DistLay &me = LAY(rank, l);
            const int sl = slot(q, id);
            auto push = [&](int dst, long long src_elem, long long dst_elem, int count) {
               DistAsyncOp p;
               memset(&p, 0, sizeof(p));
               p.type = AOP_PUSH; p.mat_kind = -1; p.mat_level = -1; p.level = l; p.barrier = 0;
               for (int r = 0; r < DROLE_N; r++) p.slot[r] = DEXT_NONE;
               p.slot[DROLE_X] = sl; p.elem[DROLE_X] = src_elem;
               p.slot[DROLE_Y] = sl; p.elem[DROLE_Y] = dst_elem;
               p.dst_rank = dst; p.count = count;      // (count 0: no such neighbour -- kept so that every rank's program has the same shape)
               p.red_scale = 1.0;
               out.ops.push_back(p);
            };
            auto sync = [&](int type, int peer, int flag) {
               DistAsyncOp p;
               memset(&p, 0, sizeof(p));
               p.type = type; p.mat_kind = -1; p.mat_level = -1; p.level = l;
               for (int r = 0; r < DROLE_N; r++) p.slot[r] = DEXT_NONE;
               p.dst_rank = peer;
               if (type == AOP_SIGNAL) p.count = flag; else p.barrier = flag;
               p.red_scale = 1.0;
               out.ops.push_back(p);
            };
            // one EXCHANGE STEP: stores, then "my stores of step s are in place" to every peer that received some, then wait
            // for the same word from every peer this rank receives from.  Inside a level group the ranks therefore move in
            // lock step, like the ranks of a grid's communicator inside the reference's ParCSR matvecs; the groups stay
            // asynchronous to one another.  (Peers that do not exist keep their place with dst_rank = -1: every rank's
            // program has the same shape.)
            if (w == 0 && gather) {
               for (int j = 1; j < nranks; j++) push((rank + j) % nranks, me.row_start, me.row_start, me.n_owned);
               for (int j = 1; j < nranks; j++) sync(AOP_SIGNAL, (rank + j) % nranks, j == 1);
               for (int j = 1; j < nranks; j++) sync(AOP_WAIT, (rank + j) % nranks, j == nranks - 1);
            } else if (l < num_dist && read_by_spmv(id)) {
               if (rank > 0) push(rank - 1, me.halo_lo, LAY(rank - 1, l).halo_lo + LAY(rank - 1, l).n_owned, me.send_lo);
               else push(-1, 0, 0, 0);
               if (rank < nranks - 1) push(rank + 1, me.halo_lo + me.n_owned - me.send_hi, 0, me.send_hi);
               else push(-1, 0, 0, 0);
               sync(AOP_SIGNAL, rank > 0 ? rank - 1 : -1, 1);
               sync(AOP_SIGNAL, rank < nranks - 1 ? rank + 1 : -1, 0);
               sync(AOP_WAIT, rank > 0 ? rank - 1 : -1, 0);
               sync(AOP_WAIT, rank < nranks - 1 ? rank + 1 : -1, 1);
            }
         }
      }
   }
   out.op_begin[L] = (int)out.ops.size();
   return AMGB_OK;
}

// Host-only probe for the CPU test suite (no CUDA call): the plan of `rank`.  layouts: nranks x num_levels x 8 ints
// (n_global, row_start, n_owned, halo_lo, halo_hi, distributed, send_lo, send_hi).  ops: max_ops DistAsyncOp; op_begin[num_levels + 1];
// slot_off[max_slots + 1] (doubles); slot_group / slot_vec [max_slots].
extern "C" int amgb_dist_async_plan(const amgb_options *o, int num_levels, int nranks, int rank, const int *layouts, int symmetric, int fact0,
                                    void *ops, int max_ops, int *op_begin, long long *slot_off, int *slot_group, int *slot_vec, int max_slots,
                                    int *num_slots)
{
   if (!o || !layouts || !ops || !op_begin || !slot_off || !slot_group || !slot_vec || !num_slots) return AMGB_EINVAL;
   static_assert(sizeof(DistLay) == 8 * sizeof(int), "DistLay is 8 ints");
   DistAsyncPlan pl;
   int rc = dist_async_plan(*o, num_levels, nranks, rank, reinterpret_cast<const DistLay *>(layouts), symmetric != 0, fact0 != 0, pl);
   if (rc) return rc;
   const int ns = (int)pl.slot_group.size();
   if ((int)pl.ops.size() > max_ops || ns > max_slots) return AMGB_ENOMEM;
   memcpy(ops, pl.ops.data(), sizeof(DistAsyncOp) * pl.ops.size());
   for (int l = 0; l <= num_levels; l++) op_begin[l] = pl.op_begin[l];
   for (int s = 0; s <= ns; s++) slot_off[s] = pl.slot_off[s];
   for (int s = 0; s < ns; s++) { slot_group[s] = pl.slot_group[s]; slot_vec[s] = pl.slot_vec[s]; }
   *num_slots = ns;
   return AMGB_OK;
}

// ---- device side --------------------------------------------------------------------------------------------------------
static_assert(sizeof(DistAsyncOp) == 200, "DistAsyncOp is mirrored by solver.py");

struct DistAsync {
   DistAsyncPlan plan;
   double *arena = nullptr;                 // this rank's slots
   std::vector<double *> base;              // [nranks]: every rank's arena as seen from here (own: arena)
   std::vector<long long> group_r0, group_ul;   // per group: slot offsets (doubles) of R(0) and UL, -1 if the group has none
   long long flag_off = 0;                  // doubles: where the exchange flags start in every rank's arena
   size_t flag_words = 0;
   double *u_save = nullptr;                // level-0 layout: the solution across the balancing launches
   bool ready = false, balanced = false;
   bool peer_timeout = false;               // a level group gave up waiting for a peer's exchange step
   bool launch_failed = false;              // this rank's cooperative launch failed (message in ctx->err)
   long long pushed_doubles_per_iteration = 0;
};

void amgb_dist_async_teardown(amgb_ctx *c)
{
   if (!c || !c->dist || !c->dist->da) return;
   DistAsync *a = c->dist->da;
   for (size_t p = 0; p < a->base.size(); p++)
      if (a->base[p] && a->base[p] != a->arena) cudaIpcCloseMemHandle(a->base[p]);
   delete a;
   c->dist->da = nullptr;
}

#ifdef AMG_HAVE_NCCL
static int dist_async_prepare(amgb_ctx *c)
{
   DistState *d = c->dist;
   if (d->da && d->da->ready) return AMGB_OK;
   if (d->da) return amgb_fail(c, AMGB_ESTATE, "an earlier preparation of the row-partitioned asynchronous solve failed on this context");
   if (c->async_ready) return amgb_fail(c, AMGB_ESTATE, "this context already ran the single-GPU asynchronous solve");
   const int L = c->L, P = d->nranks, rank = d->rank;
   const amgb_options &o = c->opt;
   int rc;
   // ---- everybody's level layouts (the peers' ghost slots are addressed from them)
   std::vector<DistLay> mine(L), all((size_t)P * L);
   for (int l = 0; l < L; l++) {
      const DistLevel &v = d->lv[l];
      mine[l] = DistLay{v.n_global, v.row_start, v.n_owned, v.halo_lo, v.halo_hi, v.distributed, v.send_lo, v.send_hi};
   }
   int *d_lay = nullptr;
   const size_t lay_ints = (size_t)L * 8;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&d_lay, sizeof(int) * lay_ints * (size_t)(P + 1), true))) return rc;
   CUDA_OK(c, cudaMemcpyAsync(d_lay + lay_ints * P, mine.data(), sizeof(int) * lay_ints, cudaMemcpyHostToDevice, c->stream));
   NCCL_OK(c, ncclAllGather(d_lay + lay_ints * P, d_lay, lay_ints, ncclInt, d->comm, c->stream));
   CUDA_OK(c, cudaMemcpyAsync(all.data(), d_lay, sizeof(int) * lay_ints * P, cudaMemcpyDeviceToHost, c->stream));
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   if (memcmp(&all[(size_t)rank * L], mine.data(), sizeof(DistLay) * L) != 0) return amgb_fail(c, AMGB_ENCCL, "layout all-gather returned another rank's table in this rank's place");
   // ---- plan
   DistAsync *a = new DistAsync();
   d->da = a;
   const bool multadd = o.solver == AMGB_SOLVER_MULTADD || o.solver == AMGB_SOLVER_ASYNC_MULTADD;
   const bool fact0 = o.factor_level0 && multadd && c->symmetric && L >= 2;
   amgb_options oa = o;
   if ((rc = dist_async_plan(oa, L, P, rank, all.data(), c->symmetric, fact0, a->plan)))
      return amgb_fail(c, rc, "the row-partitioned asynchronous solve runs Multadd or AFACx with weighted / L1 Jacobi, default asynchronous options, on consistent layouts");
   const DistAsyncPlan &pl = a->plan;
   const int ns = (int)pl.slot_group.size();
   const size_t flag_words = (size_t)L * P + 32;
   const size_t arena_bytes = sizeof(double) * ((size_t)pl.slot_off[ns] + flag_words);
   a->flag_off = pl.slot_off[ns]; a->flag_words = flag_words;
   {
      cudaError_t e = cudaMalloc((void **)&a->arena, std::max<size_t>(arena_bytes, 256));      // (its own allocation: the IPC handle maps an allocation's base)
      if (e != cudaSuccess) return amgb_fail(c, AMGB_ENOMEM, "cudaMalloc(%zu bytes) for the asynchronous vectors: %s", arena_bytes, cudaGetErrorString(e));
      c->allocs.push_back((void *)a->arena);
      c->bytes_allocated += arena_bytes;
      CUDA_OK(c, cudaMemsetAsync(a->arena, 0, std::max<size_t>(arena_bytes, 256), c->stream));
   }
   // ---- every rank's arena mapped here (CUDA IPC; the handles travel through one all-gather)
   a->base.assign(P, nullptr);
   a->base[rank] = a->arena;
   if (P > 1) {
      static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t size");
      cudaIpcMemHandle_t h;
      CUDA_OK(c, cudaIpcGetMemHandle(&h, a->arena));
      unsigned char *d_h = nullptr;
      if ((rc = amgb_dev_alloc_bytes(c, (void **)&d_h, 64 * (size_t)(P + 1), true))) return rc;
      CUDA_OK(c, cudaMemcpyAsync(d_h + 64 * (size_t)P, &h, 64, cudaMemcpyHostToDevice, c->stream));
      NCCL_OK(c, ncclAllGather(d_h + 64 * (size_t)P, d_h, 64, ncclChar, d->comm, c->stream));
      std::vector<unsigned char> hs(64 * (size_t)P);
      CUDA_OK(c, cudaMemcpyAsync(hs.data(), d_h, hs.size(), cudaMemcpyDeviceToHost, c->stream));
      CUDA_OK(c, cudaStreamSynchronize(c->stream));
      for (int p = 0; p < P; p++) {
         if (p == rank) continue;
         cudaIpcMemHandle_t hp;
         memcpy(&hp, hs.data() + 64 * (size_t)p, 64);
         void *ptr = nullptr;
         CUDA_OK(c, cudaIpcOpenMemHandle(&ptr, hp, cudaIpcMemLazyEnablePeerAccess));
         a->base[p] = (double *)ptr;
      }
   }
   // ---- device programs: operands resolved to pointers; pushes without a destination dropped
   auto ptr_of = [&](int p, int slot, long long elem) -> double * {
      if (slot == DEXT_NONE) return nullptr;
      if (slot == DEXT_F) return d->f + elem;
      if (slot == DEXT_U) return d->u + elem;
      if (slot <= DEXT_WS0) return d->ws[DEXT_WS0 - slot] + elem;
      return a->base[p] + pl.slot_off[slot] + elem;
   };
   std::vector<AsyncOp> dev_ops;
   std::vector<int> op_begin(L + 1, 0);
   a->group_r0.assign(L, -1); a->group_ul.assign(L, -1);
   for (int s = 0; s < ns; s++) {
      if (pl.slot_vec[s] == AV_ID(AV_R, 0)) a->group_r0[pl.slot_group[s]] = pl.slot_off[s];
      if (pl.slot_vec[s] == AV_ID(AV_UL, 0)) a->group_ul[pl.slot_group[s]] = pl.slot_off[s];
   }
   std::vector<double> work(L, 0.0);
   for (int q = 0; q < L; q++) {
      op_begin[q] = (int)dev_ops.size();
      long long pushed = 0;
      for (int i = pl.op_begin[q]; i < pl.op_begin[q + 1]; i++) {
         const DistAsyncOp &s = pl.ops[i];
         AsyncOp t;
         memset(&t, 0, sizeof(t));
         t.e = SpmvEpilogue();
         t.type = s.type; t.mat_kind = s.mat_kind; t.mat_level = s.mat_level; t.sval = s.sval; t.barrier = s.barrier; t.level = s.level;
         if (s.type == AOP_SIGNAL || s.type == AOP_WAIT) {
            // flag[q * P + src] of the receiving rank; an operation without a peer is kept only where it carries the step
            // counter (first signal) or the closing barrier (last wait)
            const bool keep = s.type == AOP_SIGNAL ? s.count != 0 : s.barrier != 0;
            if (s.dst_rank < 0 && !keep) continue;
            double *flags_here = a->arena + pl.slot_off[ns];
            if (s.type == AOP_SIGNAL) {
               t.zero = s.count;
               t.y = s.dst_rank < 0 ? nullptr : a->base[s.dst_rank] + pl.slot_off[ns] + ((size_t)q * P + rank);
            } else {
               t.x = s.dst_rank < 0 ? nullptr : flags_here + ((size_t)q * P + s.dst_rank);
            }
            dev_ops.push_back(t);
            continue;
         }
         if (s.type == AOP_PUSH) {
            if (s.count <= 0 || s.dst_rank < 0) continue;
            t.x = ptr_of(rank, s.slot[DROLE_X], s.elem[DROLE_X]);
            t.y = ptr_of(s.dst_rank, s.slot[DROLE_Y], s.elem[DROLE_Y]);
            t.sweeps = s.count;
            pushed += s.count;
            dev_ops.push_back(t);
            continue;
         }
         t.e.alpha = s.alpha; t.e.beta = s.beta; t.e.gamma = s.gamma; t.e.beta2 = s.beta2; t.e.xself = s.xself; t.e.red_scale = s.red_scale;
         t.x = ptr_of(rank, s.slot[DROLE_X], s.elem[DROLE_X]);
         t.y = ptr_of(rank, s.slot[DROLE_Y], s.elem[DROLE_Y]);
         t.e.b = ptr_of(rank, s.slot[DROLE_B], s.elem[DROLE_B]);
         t.e.c = ptr_of(rank, s.slot[DROLE_C], s.elem[DROLE_C]);
         t.e.rs = ptr_of(rank, s.slot[DROLE_RS], s.elem[DROLE_RS]);
         t.e.b2 = ptr_of(rank, s.slot[DROLE_B2], s.elem[DROLE_B2]);
         t.e.xs = ptr_of(rank, s.slot[DROLE_XS], s.elem[DROLE_XS]);
         t.e.red = ptr_of(rank, s.slot[DROLE_RED], s.elem[DROLE_RED]);
         t.e.red_copy = ptr_of(rank, s.slot[DROLE_RED_COPY], s.elem[DROLE_RED_COPY]);
         t.e.acc = ptr_of(rank, s.slot[DROLE_ACC], s.elem[DROLE_ACC]);
         dev_ops.push_back(t);
         if (s.type == AOP_SPMV) {
            const DevCSR &M = s.mat_kind == AMGB_MAT_A ? c->A[s.mat_level] : (s.mat_kind == AMGB_MAT_P ? c->P[s.mat_level] : (s.mat_kind == AMGB_MAT_R ? c->R[s.mat_level] : c->Ainv));
            auto it = c->sell_entries.find(&M);
            work[q] += async_op_cost(M, it == c->sell_entries.end() ? 0 : it->second) + 24.0 * M.nrows;
         } else if (s.type != AOP_COUNT_STOP) work[q] += 24.0 * c->A[s.level].nrows;
      }
      a->pushed_doubles_per_iteration += pushed;
   }
   op_begin[L] = (int)dev_ops.size();
   // ---- the persistent kernel's parameter block (as async_prepare of async.cu; the matrices are this rank's row blocks)
   AsyncParams hp;
   memset(&hp, 0, sizeof(hp));
   hp.num_levels = L;
   hp.first_group = 0;
   hp.smoother = o.smoother;
   hp.jgs_block_rows = o.jgs_block_rows;
   hp.n0 = c->A[0].nrows;
   for (int l = 0; l < L; l++) {
      hp.A[l] = c->A[l];
      if (l < L - 1) { hp.P[l] = c->P[l]; hp.R[l] = c->R[l]; }
   }
   hp.Ainv = c->Ainv;
   AsyncOp *d_ops = nullptr;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&d_ops, sizeof(AsyncOp) * std::max<size_t>(dev_ops.size(), 1), false))) return rc;
   CUDA_OK(c, cudaMemcpyAsync(d_ops, dev_ops.data(), sizeof(AsyncOp) * dev_ops.size(), cudaMemcpyHostToDevice, c->stream));
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   hp.ops = d_ops;
   for (int q = 0; q <= L; q++) hp.op_begin[q] = op_begin[q];
   c->async_work = work;
   c->async_heavy = false;
   c->async_first = 0;
   int grid = async_max_grid(kABlock, false);
   grid = std::max(L, std::min(grid, hp.n0 / 64 + L));
   if (grid < L) return amgb_fail(c, AMGB_ECUDA, "cooperative grid %d smaller than the number of level groups %d", grid, L);
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
   hp.u = d->u + d->lv[0].off();
   if (o.l2_persist && c->arena_used > 0) {
      c->window.base_ptr = c->arena;
      c->window.num_bytes = std::min(c->arena_used, c->max_window);
      c->window.hitRatio = 1.0f;
      c->window.hitProp = cudaAccessPropertyPersisting;
      c->window.missProp = cudaAccessPropertyStreaming;
      c->window_valid = true;
   }
   c->async_host = new AsyncParams(hp);
   if ((rc = amgb_dev_alloc_bytes(c, &c->async_params_dev, sizeof(AsyncParams), false))) return rc;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&a->u_save, sizeof(double) * (size_t)d->lv[0].n_ext(), true))) return rc;
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   a->ready = true;
   return AMGB_OK;
}

// one launch of the persistent kernel on this rank from the resident f, u: global r0 (collective: doubles as the barrier
// that separates this launch's ghost stores from the previous launch's), every group's copies, the kernel
static int dist_async_run(amgb_ctx *c, int num_cycles, double *r0_out, double *seconds)
{
   DistState *d = c->dist;
   DistAsync *a = d->da;
   AsyncParams &hp = *c->async_host;
   const DistLevel &L0 = d->lv[0];
   const size_t next = (size_t)L0.n_ext();
   int rc;
   hp.num_cycles = num_cycles;
   hp.converge_type = AMGB_CONVERGE_LOCAL;
   if ((rc = dist_residual(c))) return rc;                      // (leaves the ghosts of u exchanged)
   double ss;
   if ((rc = amgb_fetch_scalar(c, &ss))) return rc;
   if (r0_out) *r0_out = sqrt(ss);
   if ((rc = dist_halo(c, 0, d->r[0]))) return rc;               // every group starts from r0 WITH its ghosts, and from u
   for (int q = 0; q < c->L; q++) {
      if (a->group_r0[q] >= 0) CUDA_OK(c, cudaMemcpyAsync(a->arena + a->group_r0[q], d->r[0], sizeof(double) * next, cudaMemcpyDeviceToDevice, c->stream));
      if (a->group_ul[q] >= 0) CUDA_OK(c, cudaMemcpyAsync(a->arena + a->group_ul[q], d->u, sizeof(double) * next, cudaMemcpyDeviceToDevice, c->stream));
   }
   CUDA_OK(c, cudaMemsetAsync(hp.barrier_count, 0, sizeof(unsigned int) * AMGB_MAX_LEVELS, c->stream));
   CUDA_OK(c, cudaMemsetAsync((void *)hp.barrier_gen, 0, sizeof(unsigned int) * AMGB_MAX_LEVELS, c->stream));
   CUDA_OK(c, cudaMemsetAsync(hp.num_correct, 0, sizeof(int) * AMGB_MAX_LEVELS, c->stream));
   CUDA_OK(c, cudaMemsetAsync(hp.group_stop, 0, sizeof(int) * AMGB_MAX_LEVELS, c->stream));
   CUDA_OK(c, cudaMemsetAsync((void *)hp.converge_flag, 0, sizeof(int) * 4, c->stream));
   CUDA_OK(c, cudaMemsetAsync(hp.lock, 0, sizeof(int) * 4, c->stream));
   CUDA_OK(c, cudaMemsetAsync(hp.group_ns, 0, sizeof(unsigned long long) * AMGB_MAX_LEVELS, c->stream));
   CUDA_OK(c, cudaMemsetAsync(a->arena + a->flag_off, 0, sizeof(double) * a->flag_words, c->stream));      // exchange flags: step 0
   CUDA_OK(c, cudaMemcpyAsync(c->async_params_dev, &hp, sizeof(AsyncParams), cudaMemcpyHostToDevice, c->stream));
   // (a second collective: no rank's kernel may store into a peer whose group copies above are still being written)
   NCCL_OK(c, ncclAllReduce(c->d_scalars + 1, c->d_scalars + 1, 1, ncclDouble, ncclSum, d->comm, c->stream));
   d->collectives++;
   CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
   const int lr = launch_async(c->stream, (const AsyncParams *)c->async_params_dev, c->async_grid_used, kABlock, false,
                               c->window_valid ? &c->window : nullptr);
   if (lr < 0) {
      // (no early return: the peers' kernels are waiting for this rank's exchange steps and will give up after 30 s; the
      //  failure is reported once the ranks have agreed on it, so that nobody is left alone inside a collective)
      amgb_fail(c, AMGB_ECUDA, "cooperative launch failed: %s", cudaGetErrorString((cudaError_t)(-lr)));
      a->peer_timeout = true;
      a->launch_failed = true;
      return AMGB_OK;
   }
   c->launches += 1;
   CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
   {
      // (bounded wait: a persistent kernel that never returns must fail the call, not hang the job)
      const double t_start = omp_get_wtime();
      cudaError_t q;
      while ((q = cudaEventQuery(c->ev1)) == cudaErrorNotReady)
         if (omp_get_wtime() - t_start > 120.0) return amgb_fail(c, AMGB_ECUDA, "the persistent kernel did not finish within 120 s");
      CUDA_OK(c, q);
   }
   float ms = 0;
   cudaEventElapsedTime(&ms, c->ev0, c->ev1);
   if (seconds) *seconds = ms * 1e-3;
   int flags[4] = {0, 0, 0, 0};
   CUDA_OK(c, cudaMemcpy(flags, (const void *)hp.converge_flag, sizeof(flags), cudaMemcpyDeviceToHost));
   if (flags[1]) a->peer_timeout = true;      // (reported after the ranks have agreed on it: the call stays collective)
   d->halo_bytes += 8LL * a->pushed_doubles_per_iteration * num_cycles;
   CUDA_OK(c, cudaGetLastError());
   return AMGB_OK;
}
#endif   // AMG_HAVE_NCCL

#ifdef AMG_HAVE_NCCL
// every rank learns whether ANY rank's launch failed or timed out waiting for a peer, and all of them fail together
static int dist_async_agree(amgb_ctx *c)
{
   DistState *d = c->dist;
   DistAsync *a = d->da;
   const double mine = a->peer_timeout ? 1.0 : 0.0;
   CUDA_OK(c, cudaMemcpyAsync(c->d_scalars + 2, &mine, sizeof(double), cudaMemcpyHostToDevice, c->stream));
   NCCL_OK(c, ncclAllReduce(c->d_scalars + 2, c->d_scalars + 2, 1, ncclDouble, ncclMax, d->comm, c->stream));
   double any = 0.0;
   CUDA_OK(c, cudaMemcpyAsync(&any, c->d_scalars + 2, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   const bool was_mine = a->launch_failed;
   a->peer_timeout = false;
   a->launch_failed = false;
   if (any != 0.0) {
      if (was_mine) return AMGB_ECUDA;                    // (keep this rank's own message: the launch failure)
      return amgb_fail(c, AMGB_ENCCL, "a level group waited 30 s for a peer GPU's exchange step (a peer's kernel was not running): the solve is void");
   }
   return AMGB_OK;
}
#endif

// Asynchronous additive solve on the partitioned hierarchy from the resident f and u (amgb_dist_set_rhs; u = 0 after
// amgb_dist_setup / amgb_dist_zero_solution): every level group of every rank performs num_cycles corrections (LOCAL stop
// rule).  Collective.  corrections[num_levels]: this rank's counts; relres: global ||f - A u|| / ||f - A u_start||;
// solve_seconds: this rank's kernel time (the job's time is the maximum over the ranks).
extern "C" int amgb_dist_solve_async(amgb_ctx *c, int num_cycles, int *corrections, double *relres, double *solve_seconds)
{
   NEED_READY(c);
#ifdef AMG_HAVE_NCCL
   DistState *d = c->dist;
   if (!d || !d->ready) return amgb_fail(c, AMGB_ESTATE, "amgb_dist_setup not called");
   if (num_cycles < 1) return amgb_fail(c, AMGB_EINVAL, "num_cycles < 1");
   if (c->opt.solver == AMGB_SOLVER_MULT) return amgb_fail(c, AMGB_EINVAL, "there is no asynchronous MULT: DMEM_Add_async runs Multadd or AFACx");
   if (c->opt.coarse_solve && c->L > 1 && !c->Ainv.rp) return amgb_fail(c, AMGB_ESTATE, "coarse_solve: the inverse of the coarsest operator was not built");
   int rc;
   if ((rc = dist_async_prepare(c))) return rc;
   DistAsync *a = d->da;
   AsyncParams &hp = *c->async_host;
   const int L = c->L;
   const size_t next = (size_t)d->lv[0].n_ext();
   if (!a->balanced) {
      // CTA groups from measured group times, as on one GPU (amgb_solve_async): two short launches, u restored afterwards.
      // Every rank sizes its own groups; all ranks run the same number of launches (each launch is collective).
      async_assign_groups(c, c->async_work);
      const char *env = getenv("AMGB_ASYNC_BALANCE");
      const int rounds = env ? atoi(env) : 2;
      if (rounds > 0 && L > 2) {
         CUDA_OK(c, cudaMemcpyAsync(a->u_save, d->u, sizeof(double) * next, cudaMemcpyDeviceToDevice, c->stream));
         for (int it = 0; it < rounds; it++) {
            if ((rc = dist_async_run(c, 3, nullptr, nullptr))) return rc;
            if ((rc = dist_async_agree(c))) return rc;
            std::vector<unsigned long long> ns(AMGB_MAX_LEVELS);
            CUDA_OK(c, cudaMemcpy(ns.data(), hp.group_ns, sizeof(unsigned long long) * AMGB_MAX_LEVELS, cudaMemcpyDeviceToHost));
            std::vector<double> work(AMGB_MAX_LEVELS, 0.0);
            for (int q = 0; q < L; q++) {
               const int nct = hp.cta_begin[q + 1] - hp.cta_begin[q];
               work[q] = c->async_work[q] > 0.0 ? (double)nct * (double)ns[q] : 0.0;
            }
            // the ranks of one level group move in lock step, so a group is as fast as its slowest rank: every rank deals
            // its CTAs from the SUM over the ranks (the same split everywhere)
            static_assert(AMGB_MAX_LEVELS + 8 <= 64, "d_scalars holds 64 doubles");
            CUDA_OK(c, cudaMemcpyAsync(c->d_scalars + 8, work.data(), sizeof(double) * AMGB_MAX_LEVELS, cudaMemcpyHostToDevice, c->stream));
            NCCL_OK(c, ncclAllReduce(c->d_scalars + 8, c->d_scalars + 8, AMGB_MAX_LEVELS, ncclDouble, ncclSum, d->comm, c->stream));
            CUDA_OK(c, cudaMemcpyAsync(work.data(), c->d_scalars + 8, sizeof(double) * AMGB_MAX_LEVELS, cudaMemcpyDeviceToHost, c->stream));
            CUDA_OK(c, cudaStreamSynchronize(c->stream));
            work.resize(L);
            async_assign_groups(c, work);
            CUDA_OK(c, cudaMemcpyAsync(d->u, a->u_save, sizeof(double) * next, cudaMemcpyDeviceToDevice, c->stream));
         }
      }
      a->balanced = true;
   }
   double r0 = 0.0;
   if ((rc = dist_async_run(c, num_cycles, &r0, solve_seconds))) return rc;
   if ((rc = dist_async_agree(c))) return rc;
   if ((rc = dist_residual(c))) return rc;
   double ss;
   if ((rc = amgb_fetch_scalar(c, &ss))) return rc;
   if (relres) *relres = r0 > 0.0 ? sqrt(ss) / r0 : 0.0;
   c->r0_norm = r0;
   if (corrections) {
      std::vector<int> h(AMGB_MAX_LEVELS);
      CUDA_OK(c, cudaMemcpy(h.data(), hp.num_correct, sizeof(int) * AMGB_MAX_LEVELS, cudaMemcpyDeviceToHost));
      for (int l = 0; l < L; l++) corrections[l] = h[l];
   }
   CUDA_OK(c, cudaGetLastError());
   return AMGB_OK;
#else
   (void)num_cycles; (void)corrections; (void)relres; (void)solve_seconds;
   return amgb_fail(c, AMGB_ENCCL, "library built without NCCL");
#endif
}

// CTA groups of the last launch and the seconds every group spent in it (this rank)
extern "C" int amgb_dist_async_groups(amgb_ctx *c, int *cta_begin /* num_levels + 1 */, double *seconds /* num_levels */)
{
   NEED_READY(c);
   if (!c->dist || !c->dist->da || !c->dist->da->ready) return amgb_fail(c, AMGB_ESTATE, "no row-partitioned asynchronous solve yet");
   std::vector<unsigned long long> ns(AMGB_MAX_LEVELS);
   CUDA_OK(c, cudaMemcpy(ns.data(), c->async_host->group_ns, sizeof(unsigned long long) * AMGB_MAX_LEVELS, cudaMemcpyDeviceToHost));
   for (int l = 0; l < c->L; l++) {
      if (cta_begin) cta_begin[l] = c->async_host->cta_begin[l];
      if (seconds) seconds[l] = 1e-9 * (double)ns[l];
   }
   if (cta_begin) cta_begin[c->L] = c->async_host->cta_begin[c->L];
   return AMGB_OK;
}

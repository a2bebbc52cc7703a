// dist.cu -- multi-GPU synchronous additive solve: one process per GPU, rows of every level partitioned
// contiguously, NCCL over NVLink for the halo exchange, the coarse all-gather and the norms.
//
// Replaces, for the synchronous Multadd cycle, the reference's DMEM path: DMEM_Add / DMEM_SyncAdd
// (src/DMEM_Add.cpp:20-178, src/DMEM_Mult.cpp:263-450), whose distributed SpMVs are hypre ParCSR matvecs
// (halo exchange through hypre's comm_pkg, src/DMEM_Add.cpp:230-249,277-308) and whose vector traffic
// goes through DMEM_Comm's MPI engine (src/DMEM_Comm.cpp:81-382); the residual norm is an Allreduce
// (src/DMEM_Misc.cpp:398-433).
//
// Layout (host logic in async-multigrid_b200/partition.py): a DISTRIBUTED level's vectors live in the
// rank's extended index space [ghost_lo | owned | ghost_hi]; the local row blocks of A_l, P_l, R_l carry
// column indices in that space, so the SpMV kernels are the single-GPU ones and a halo exchange is two
// contiguous ncclSend/ncclRecv pairs with the immediate neighbours, no packing.  REPLICATED levels (the
// small coarse tail) hold full vectors and matrices on every rank; the first replicated level's
// residual is all-gathered, everything coarser is computed redundantly with no communication.
#include "dist.h"
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>
#include <omp.h>

void amgb_dist_teardown(amgb_ctx *c)
{
   if (c && c->dist) {
      amgb_dist_async_teardown(c);
#ifdef AMG_HAVE_NCCL
      if (c->dist->comm) ncclCommDestroy(c->dist->comm);
#endif
      if (c->dist->graph_exec) cudaGraphExecDestroy(c->dist->graph_exec);
      if (c->dist->nbr_lo) cudaIpcCloseMemHandle(c->dist->nbr_lo);
      if (c->dist->nbr_hi) cudaIpcCloseMemHandle(c->dist->nbr_hi);
      if (c->dist->comm_stream) cudaStreamDestroy(c->dist->comm_stream);
      if (c->dist->ev_x) cudaEventDestroy(c->dist->ev_x);
      if (c->dist->ev_h) cudaEventDestroy(c->dist->ev_h);
      delete c->dist;
      c->dist = nullptr;
   }
}

int amgb_dist_diag_offset(const amgb_ctx *c, int level)
{
   if (!c->dist || level >= (int)c->dist->lv.size() || !c->dist->lv[level].set) return 0;
   return c->dist->lv[level].off();
}
bool amgb_dist_owned_cols(const amgb_ctx *c, int kind, int level, int *c0, int *c1)
{
   if (!c->dist) return false;
   const int in = kind == AMGB_MAT_P ? level + 1 : level;      // level of the matrix's input vector
   if (in >= (int)c->dist->lv.size() || !c->dist->lv[in].set || !c->dist->lv[in].distributed) return false;
   // the rows must be partitioned too (a replicated matrix has nothing to overlap)
   const int out = kind == AMGB_MAT_R ? level + 1 : level;
   if (kind != AMGB_MAT_R && !c->dist->lv[out].distributed) return false;
   *c0 = c->dist->lv[in].halo_lo;
   *c1 = c->dist->lv[in].halo_lo + c->dist->lv[in].n_owned;
   return true;
}

bool amgb_dist_level_distributed(const amgb_ctx *c, int level)
{
   return c->dist && level < (int)c->dist->lv.size() && c->dist->lv[level].set && c->dist->lv[level].distributed;
}

static inline SpmvEpilogue epi(double alpha, double beta, const double *b, double gamma = 0.0, const double *cc = nullptr,
                               const double *rs = nullptr)
{
   SpmvEpilogue e;
   e.alpha = alpha; e.beta = beta; e.gamma = gamma; e.b = b; e.c = cc; e.rs = rs;
   return e;
}

#ifdef AMG_HAVE_NCCL
// ghosts of v (level layout) <- neighbours' boundary entries
int dist_halo(amgb_ctx *c, int l, double *v, cudaStream_t st)
{
   DistState *d = c->dist;
   const DistLevel &L = d->lv[l];
   if (!L.distributed) return AMGB_OK;
   if (!st) st = c->stream;
   double *own = v + L.halo_lo;
   NCCL_OK(c, ncclGroupStart());
   if (d->rank > 0) {
      if (L.send_lo) NCCL_OK(c, ncclSend(own, (size_t)L.send_lo, ncclDouble, d->rank - 1, d->comm, st));
      if (L.halo_lo) NCCL_OK(c, ncclRecv(v, (size_t)L.halo_lo, ncclDouble, d->rank - 1, d->comm, st));
   }
   if (d->rank < d->nranks - 1) {
      if (L.send_hi) NCCL_OK(c, ncclSend(own + L.n_owned - L.send_hi, (size_t)L.send_hi, ncclDouble, d->rank + 1, d->comm, st));
      if (L.halo_hi) NCCL_OK(c, ncclRecv(own + L.n_owned, (size_t)L.halo_hi, ncclDouble, d->rank + 1, d->comm, st));
   }
   NCCL_OK(c, ncclGroupEnd());
   d->halo_bytes += 8LL * (L.send_lo + L.send_hi);
   d->collectives++;
   return AMGB_OK;
}

// every rank's owned slice of a replicated vector -> everybody (in place)
static int allgather_level(amgb_ctx *c, int l, double *v)
{
   DistState *d = c->dist;
   const DistLevel &L = d->lv[l];
   NCCL_OK(c, ncclGroupStart());
   size_t off = 0;
   for (int p = 0; p < d->nranks; p++) {
      const size_t cnt = (size_t)L.all_owned[p];
      if (cnt) NCCL_OK(c, ncclBroadcast(v + off, v + off, cnt, ncclDouble, p, d->comm, c->stream));
      off += cnt;
   }
   NCCL_OK(c, ncclGroupEnd());
   d->collectives++;
   return AMGB_OK;
}

// y = epilogue(M x) where x (level `lin` layout, owned part final on the main stream) still needs its ghosts:
// the exchange runs on the communication stream while the launch units that read only owned entries run on
// the main stream; the boundary units follow once the ghosts have landed.  (The reference overlaps the same
// way inside hypre's ParCSR matvec: diag block while the comm_pkg exchange is in flight, then the offd block;
// its own attempt is at src/DMEM_Smooth.cpp:205-214.)
static int dist_spmv(amgb_ctx *c, const DevCSR &M, bool sval, int lin, double *x, double *y, const SpmvEpilogue &e, bool norm)
{
   DistState *d = c->dist;
   int rc;
   const bool split = d->overlap && d->lv[lin].distributed && M.uhi > M.ulo;
   if (!split) {
      if ((rc = dist_halo(c, lin, x))) return rc;
      enq_spmv(c, M, sval, x, y, e, norm);
      return AMGB_OK;
   }
   CUDA_OK(c, cudaEventRecord(d->ev_x, c->stream));
   CUDA_OK(c, cudaStreamWaitEvent(d->comm_stream, d->ev_x, 0));
   if ((rc = dist_halo(c, lin, x, d->comm_stream))) return rc;
   CUDA_OK(c, cudaEventRecord(d->ev_h, d->comm_stream));
   const int nu = spmv_units(M), np = c->npartials;
   int g0 = 0, g1 = 0, g2 = 0;
   if (norm) CUDA_OK(c, cudaMemsetAsync(d->partials3, 0, sizeof(double) * 3 * np, c->stream));
   c->launches += launch_spmv_units(c->cfg, c->stream, M, M.ulo, M.uhi, sval, x, y, e, norm ? d->partials3 : nullptr, &g0);
   CUDA_OK(c, cudaStreamWaitEvent(c->stream, d->ev_h, 0));
   c->launches += launch_spmv_units(c->cfg, c->stream, M, 0, M.ulo, sval, x, y, e, norm ? d->partials3 + np : nullptr, &g1);
   c->launches += launch_spmv_units(c->cfg, c->stream, M, M.uhi, nu, sval, x, y, e, norm ? d->partials3 + 2 * np : nullptr, &g2);
   if (norm) c->launches += launch_reduce_partials(c->stream, d->partials3, 3 * np, c->d_scalars);
   (void)g0; (void)g1; (void)g2;
   return AMGB_OK;
}

// r_0 = f - A_0 u on the owned rows, d_scalars[0] = global ||r||^2
int dist_residual(amgb_ctx *c)
{
   DistState *d = c->dist;
   int rc;
   if ((rc = dist_spmv(c, c->A[0], false, 0, d->u, d->r[0] + d->lv[0].off(), epi(-1.0, 1.0, d->f), true))) return rc;
   NCCL_OK(c, ncclAllReduce(c->d_scalars, c->d_scalars, 1, ncclDouble, ncclSum, d->comm, c->stream));
   d->collectives++;
   return AMGB_OK;
}

// one synchronous Multadd cycle on r[0]; u += B r   (SMEM_Sync_Add_Vcycle semantics, src/SEQ_AMG.cpp:110-235;
// DMEM analogue DMEM_SyncAddCycle, src/DMEM_Mult.cpp:322-450, with the SMEM convention that the coarsest
// level contributes nothing)
// tgt: owned rows of a level-0 vector; accumulate: tgt += B r, else tgt = B r
static int dist_cycle(amgb_ctx *c, double *tgt, bool accumulate)
{
   DistState *d = c->dist;
   const int L = c->L;
   int rc;
   if (L == 1) {
      if (!accumulate) CUDA_OK(c, cudaMemsetAsync(tgt, 0, sizeof(double) * c->A[0].nrows, c->stream));
      return AMGB_OK;
   }
   const bool bpx = c->opt.solver == AMGB_SOLVER_BPX;                   // SYNC_BPX of DMEM_SyncAddCycle (src/DMEM_Mult.cpp:346-349)
   const bool afacx = c->opt.solver == AMGB_SOLVER_AFACX;               // AFACx with the SMEM / SEQ meaning (src/SEQ_AMG.cpp:172-208), row-partitioned
   const bool direct = c->opt.coarse_solve && c->Ainv.rp != nullptr;   // DMEM: direct solve on the (replicated) coarsest level
   const int top = (direct || bpx) ? L : L - 1;                         // levels that contribute a correction
   const int last_r = afacx ? L - 1 : top - 1;                          // AFACx level L-2 smooths r_{L-1} on its coarse side
   // level-0 transfers in factorised form (see enq_cycle in context.cu): plain P_0 / R_0 uploaded
   const bool fact0 = c->opt.factor_level0 && c->symmetric && top >= 2;
   const int off0 = d->lv[0].off();
   for (int l = 0; l < last_r; l++) {
      const DistLevel &nx = d->lv[l + 1];
      const bool gather = d->lv[l].distributed && !nx.distributed;
      double *out = d->r[l + 1] + (gather ? nx.row_start : nx.off());
      if (fact0 && l == 0) {
         // t_0 = r_0 - A_0 diag(w/d) r_0 (ghosts of r_0), then r_1 = R_0 t_0 (ghosts of t_0)
         if ((rc = dist_spmv(c, c->A[0], true, 0, d->r[0], d->t0 + off0, epi(-1.0, 1.0, d->r[0] + off0), false))) return rc;
         if ((rc = dist_spmv(c, c->R[0], false, 0, d->t0, out, epi(1.0, 0.0, nullptr), false))) return rc;
      } else if ((rc = dist_spmv(c, c->R[l], false, l, d->r[l], out, epi(1.0, 0.0, nullptr), false))) return rc;
      if (gather && (rc = allgather_level(c, l + 1, d->r[l + 1]))) return rc;
   }
   if (top == L - 1 && c->symmetric && (rc = dist_halo(c, L - 2, d->r[L - 2]))) return rc;   // (the other smoothers read owned entries only)
   if (direct) enq_spmv(c, c->Ainv, false, d->r[L - 1], d->e[L - 1], epi(1.0, 0.0, nullptr), false);
   for (int l = 0; l < (direct ? L - 1 : top); l++) {
      if (fact0 && l == 0) continue;                  // e_0 is folded into the last launch of the cycle
      const DistLevel &lv = d->lv[l];
      const double *rown = d->r[l] + lv.off();
      const double *ws = d->ws[l] + lv.off();
      if (afacx) {
         // src/SEQ_AMG.cpp:172-208 with one sweep on either side: u_c = s_{l+1} o r_{l+1};  e = P_l u_c (ghosts of u_c);
         // r_f = r_l - A_l e (ghosts of e);  u_f = s_l o r_f
         const DistLevel &nx = d->lv[l + 1];
         c->launches += launch_scale(c->cfg, c->stream, c->A[l + 1].nrows, d->ws[l + 1] + nx.off(), d->r[l + 1] + nx.off(), d->t[l + 1] + nx.off());
         if ((rc = dist_spmv(c, c->P[l], false, l + 1, d->t[l + 1], d->w[l] + lv.off(), epi(1.0, 0.0, nullptr), false))) return rc;
         if ((rc = dist_spmv(c, c->A[l], false, l, d->w[l], d->t[l] + lv.off(), epi(-1.0, 1.0, rown), false))) return rc;
         c->launches += launch_scale(c->cfg, c->stream, c->A[l].nrows, ws, d->t[l] + lv.off(), d->e[l] + lv.off());
      } else if (c->symmetric)   // e = (w/d) o (2 r - (A diag(w/d)) r)
         enq_spmv(c, c->A[l], true, d->r[l], d->e[l] + lv.off(), epi(-1.0, 2.0, rown, 0.0, nullptr, ws), false);
      else
         c->launches += launch_scale(c->cfg, c->stream, c->A[l].nrows, ws, rown, d->e[l] + lv.off());
   }
   for (int l = top - 2; l >= 1; l--) {
      double *eo = d->e[l] + d->lv[l].off();
      if ((rc = dist_spmv(c, c->P[l], false, l + 1, d->e[l + 1], eo, epi(1.0, 1.0, eo), false))) return rc;
   }
   double *uo = tgt;
   const double *cacc = accumulate ? tgt : nullptr;
   if (fact0) {
      // v = P_0 e_1 (ghosts of e_1);  u += v + (w/d) o (r_0 + t_0 - A_0 v) (ghosts of v)
      if ((rc = dist_spmv(c, c->P[0], false, 1, d->e[1], d->v0 + off0, epi(1.0, 0.0, nullptr), false))) return rc;
      SpmvEpilogue fe = epi(-1.0, 1.0, d->r[0] + off0, 1.0, cacc, d->ws[0] + off0);
      fe.b2 = d->t0 + off0; fe.beta2 = 1.0;
      fe.xs = d->v0 + off0; fe.xself = 1.0;
      if ((rc = dist_spmv(c, c->A[0], false, 0, d->v0, uo, fe, false))) return rc;
   } else if (top >= 2) {
      if ((rc = dist_spmv(c, c->P[0], false, 1, d->e[1], uo, epi(1.0, 1.0, d->e[0] + d->lv[0].off(), 1.0, cacc), false))) return rc;
   } else if (accumulate) {
      c->launches += launch_add(c->cfg, c->stream, c->A[0].nrows, d->e[0] + d->lv[0].off(), uo);
   } else {
      CUDA_OK(c, cudaMemcpyAsync(uo, d->e[0] + d->lv[0].off(), sizeof(double) * c->A[0].nrows, cudaMemcpyDeviceToDevice, c->stream));
   }
   return AMGB_OK;
}

// `sweeps` (L1-)Jacobi sweeps u <- u + s o (f - A_l u) on level l.  u (level layout) starts in *cur, one of the level's two
// buffers a / b, and ping-pongs between them; *cur names the buffer that holds the result.  f: the level's rows.
static int dist_sweeps(amgb_ctx *c, int l, const double *f, double **cur, double *a, double *b, int sweeps)
{
   DistState *d = c->dist;
   const int off = d->lv[l].off();
   const double *s = d->ws[l] + off;
   int rc;
   for (int k = 0; k < sweeps; k++) {
      double *nxt = *cur == a ? b : a;
      if ((rc = dist_spmv(c, c->A[l], false, l, *cur, nxt + off, epi(-1.0, 1.0, f, 1.0, *cur + off, s), false))) return rc;
      *cur = nxt;
   }
   return AMGB_OK;
}

// One multiplicative V-cycle on (f, u) of level 0, row-partitioned: SMEM_Sync_Parfor_Vcycle (src/SMEM_Sync_AMG.cpp:8-145) with
// the meaning and the quirks of enq_vcycle (context.cu) -- level right-hand sides in r[l], level solutions in e[l] (l >= 1), the
// first pre-sweep of levels 1..L-2 from a zero guess, the coarsest level's num_pre + num_post sweeps continuing from what the
// previous cycle left in e[L-1], or with coarse_solve DMEM_MultCycle's direct solve there (src/DMEM_Mult.cpp:207).  Every SpMV
// that reads a distributed vector exchanges its ghosts first (dist_spmv); the restricted residual of the first replicated level
// is all-gathered as in dist_cycle.  A level's iterate ping-pongs between its home buffer and t[l]; the prolongation writes
// into whichever of the two makes the post-sweeps end in the home buffer, so only the coarsest level (whose iterate must
// persist across cycles) may need a copy.
static int dist_vcycle(amgb_ctx *c)
{
   DistState *d = c->dist;
   const int L = c->L;
   const int pre = c->opt.num_pre_smooth_sweeps, post = c->opt.num_post_smooth_sweeps;
   int rc;
   auto rhs = [&](int l) -> const double * { return l == 0 ? d->f : d->r[l] + d->lv[l].off(); };
   auto home = [&](int l) -> double * { return l == 0 ? d->u : d->e[l]; };
   std::vector<double *> down((size_t)L);                    // where each level's iterate is after the pre-smoothing
   for (int l = 0; l < L - 1; l++) {
      const DistLevel &lv = d->lv[l], &nx = d->lv[l + 1];
      const int off = lv.off();
      const double *f = rhs(l);
      double *cur = home(l);
      if (l > 0 && pre > 0) {
         // zero guess: u = s o f; with one sweep the residual f - A (s o f) comes from the column-scaled values (ghosts of f)
         c->launches += launch_scale(c->cfg, c->stream, c->A[l].nrows, d->ws[l] + off, f, cur + off);
         if (pre == 1) {
            if ((rc = dist_spmv(c, c->A[l], true, l, d->r[l], d->w[l] + off, epi(-1.0, 1.0, f), false))) return rc;
         } else {
            if ((rc = dist_sweeps(c, l, f, &cur, home(l), d->t[l], pre - 1))) return rc;
            if ((rc = dist_spmv(c, c->A[l], false, l, cur, d->w[l] + off, epi(-1.0, 1.0, f), false))) return rc;
         }
      } else {
         // level 0 continues from the current u; with no pre-sweep a coarser level keeps the previous cycle's iterate
         if ((rc = dist_sweeps(c, l, f, &cur, home(l), d->t[l], pre))) return rc;
         if ((rc = dist_spmv(c, c->A[l], false, l, cur, d->w[l] + off, epi(-1.0, 1.0, f), false))) return rc;
      }
      down[l] = cur;
      const bool gather = lv.distributed && !nx.distributed;
      double *out = d->r[l + 1] + (gather ? nx.row_start : nx.off());
      if ((rc = dist_spmv(c, c->R[l], false, l, d->w[l], out, epi(1.0, 0.0, nullptr), false))) return rc;
      if (gather && (rc = allgather_level(c, l + 1, d->r[l + 1]))) return rc;
   }
   {
      const int cl = L - 1, off = d->lv[cl].off();
      if (c->opt.coarse_solve && c->Ainv.rp) {
         enq_spmv(c, c->Ainv, false, d->r[cl], d->e[cl], epi(1.0, 0.0, nullptr), false);     // replicated level (amgb_dist_setup)
      } else {
         double *cur = home(cl);
         if ((rc = dist_sweeps(c, cl, rhs(cl), &cur, home(cl), d->t[cl], pre + post))) return rc;
         if (cur != home(cl))
            CUDA_OK(c, cudaMemcpyAsync(home(cl) + off, cur + off, sizeof(double) * c->A[cl].nrows, cudaMemcpyDeviceToDevice, c->stream));
      }
   }
   for (int l = L - 2; l >= 0; l--) {
      const int off = d->lv[l].off();
      // u_l += P_l u_{l+1} (ghosts of u_{l+1} when level l+1 is distributed), written where the post-sweeps end in home(l)
      double *cur = (post & 1) ? d->t[l] : home(l);
      if ((rc = dist_spmv(c, c->P[l], false, l + 1, home(l + 1), cur + off, epi(1.0, 1.0, down[l] + off), false))) return rc;
      if ((rc = dist_sweeps(c, l, rhs(l), &cur, home(l), d->t[l], post))) return rc;
   }
   return AMGB_OK;
}

// one iteration of the synchronous solve without acceleration: the cycle on u, then r = f - A u and its all-reduced norm
static int dist_iteration(amgb_ctx *c)
{
   int rc;
   if (c->opt.solver == AMGB_SOLVER_MULT) rc = dist_vcycle(c);
   else rc = dist_cycle(c, c->dist->u + c->dist->lv[0].off(), true);
   return rc ? rc : dist_residual(c);
}
#endif   // AMG_HAVE_NCCL

extern "C" {

int amgb_dist_unique_id(unsigned char id128[128])
{
#ifdef AMG_HAVE_NCCL
   static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
   ncclUniqueId id;
   if (ncclGetUniqueId(&id) != ncclSuccess) return AMGB_ENCCL;
   memcpy(id128, &id, 128);
   return AMGB_OK;
#else
   (void)id128;
   return AMGB_ENCCL;
#endif
}

int amgb_dist_init(amgb_ctx *c, const unsigned char id128[128], int rank, int nranks)
{
   if (!c || !id128 || nranks < 1 || rank < 0 || rank >= nranks) return amgb_fail(c, AMGB_EINVAL, "bad rank / nranks");
   if (c->dist) return amgb_fail(c, AMGB_ESTATE, "amgb_dist_init called twice");
   if (c->L) return amgb_fail(c, AMGB_ESTATE, "amgb_dist_init must precede the hierarchy upload");
#ifdef AMG_HAVE_NCCL
   CUDA_OK(c, cudaSetDevice(c->device));
   DistState *d = new DistState();
   d->rank = rank; d->nranks = nranks;
   ncclUniqueId id;
   memcpy(&id, id128, 128);
   ncclResult_t r = ncclCommInitRank(&d->comm, nranks, id, rank);
   if (r != ncclSuccess) { delete d; return amgb_fail(c, AMGB_ENCCL, "ncclCommInitRank: %s", ncclGetErrorString(r)); }
   c->dist = d;
   return AMGB_OK;
#else
   return amgb_fail(c, AMGB_ENCCL, "library built without NCCL");
#endif
}

int amgb_dist_set_level(amgb_ctx *c, int level, int n_global, int row_start, int n_owned, int halo_lo, int halo_hi,
                        int distributed, int send_lo, int send_hi, const int *all_owned)
{
   if (!c || !c->dist) return amgb_fail(c, AMGB_ESTATE, "amgb_dist_init not called");
   if (c->L == 0) return amgb_fail(c, AMGB_ESTATE, "call amgb_set_num_levels first");
   if (level < 0 || level >= c->L || n_global < 0 || n_owned < 0 || row_start < 0 || row_start + n_owned > n_global ||
       halo_lo < 0 || halo_hi < 0 || send_lo < 0 || send_hi < 0 || send_lo > n_owned || send_hi > n_owned || !all_owned)
      return amgb_fail(c, AMGB_EINVAL, "bad level layout");
   DistState *d = c->dist;
   if ((int)d->lv.size() != c->L) d->lv.resize(c->L);
   if (c->A[level].rp) return amgb_fail(c, AMGB_ESTATE, "amgb_dist_set_level must precede amgb_set_matrix for level %d", level);
   DistLevel &L = d->lv[level];
   L.n_global = n_global; L.row_start = row_start; L.n_owned = n_owned;
   L.distributed = distributed ? 1 : 0;
   L.halo_lo = distributed ? halo_lo : 0; L.halo_hi = distributed ? halo_hi : 0;
   L.send_lo = distributed ? send_lo : 0; L.send_hi = distributed ? send_hi : 0;
   L.all_owned.assign(all_owned, all_owned + d->nranks);
   long tot = 0;
   for (int v : L.all_owned) tot += v;
   if (tot != n_global || L.all_owned[d->rank] != n_owned) return amgb_fail(c, AMGB_EINVAL, "owned counts of level %d do not add up", level);
   if (level > 0 && L.distributed && !d->lv[level - 1].distributed) return amgb_fail(c, AMGB_EINVAL, "a distributed level below a replicated one");
   L.set = true;
   return AMGB_OK;
}

int amgb_dist_setup(amgb_ctx *c)
{
   NEED_READY(c);
#ifdef AMG_HAVE_NCCL
   DistState *d = c->dist;
   if (!d) return amgb_fail(c, AMGB_ESTATE, "amgb_dist_init not called");
   if (d->ready) return amgb_fail(c, AMGB_ESTATE, "amgb_dist_setup already done");
   const int L = c->L;
   const amgb_options &o = c->opt;
   const bool mult = o.solver == AMGB_SOLVER_MULT;
   if (mult && o.smoother != AMGB_SMOOTH_JACOBI && o.smoother != AMGB_SMOOTH_L1_JACOBI)
      return amgb_fail(c, AMGB_EINVAL, "partitioned MULT smooths with weighted or L1 Jacobi: smoother %d (hybrid JGS or a Gauss-Seidel "
                                       "type) is not implemented on the partitioned path", o.smoother);
   if ((o.solver != AMGB_SOLVER_MULTADD && o.solver != AMGB_SOLVER_BPX && o.solver != AMGB_SOLVER_AFACX && !mult) ||
       (o.smoother != AMGB_SMOOTH_JACOBI && o.smoother != AMGB_SMOOTH_L1_JACOBI))
      return amgb_fail(c, AMGB_EINVAL, "the partitioned path implements synchronous Multadd, AFACx, BPX and MULT with weighted or L1 Jacobi");
   if (mult && (o.num_pre_smooth_sweeps < 0 || o.num_post_smooth_sweeps < 0 || o.num_pre_smooth_sweeps + o.num_post_smooth_sweeps < 1))
      return amgb_fail(c, AMGB_EINVAL, "partitioned MULT needs num_pre_smooth_sweeps >= 0, num_post_smooth_sweeps >= 0, one of them positive");
   if (mult && (o.coarse_solve < 0 || o.coarse_solve > 1)) return amgb_fail(c, AMGB_EINVAL, "coarse_solve must be 0 or 1");
   if (o.solver == AMGB_SOLVER_BPX && o.num_pre_smooth_sweeps != 1)
      return amgb_fail(c, AMGB_EINVAL, "partitioned BPX runs one Jacobi sweep per level");
   if (o.solver == AMGB_SOLVER_AFACX && (o.num_fine_smooth_sweeps != 1 || o.num_coarse_smooth_sweeps != 1 || o.coarse_solve))
      return amgb_fail(c, AMGB_EINVAL, "partitioned AFACx runs one fine and one coarse sweep per level, SMEM coarsest-level convention");
   if (o.solver == AMGB_SOLVER_MULTADD && o.num_fine_smooth_sweeps != 1)
      return amgb_fail(c, AMGB_EINVAL, "partitioned Multadd runs one smoothing sweep per level");
   const bool l1s = o.smoother == AMGB_SMOOTH_L1_JACOBI;
   if ((int)d->lv.size() != L) return amgb_fail(c, AMGB_ESTATE, "level layouts missing");
   // (amgb_set_matrix builds no inverse of a partitioned row block)
   if (o.coarse_solve && L > 1 && d->lv[L - 1].distributed)
      return amgb_fail(c, AMGB_EINVAL, "coarse_solve (direct coarsest solve) needs a replicated coarsest level; level %d is distributed", L - 1);
   int rc;
   for (int l = 0; l < L; l++) {
      const DistLevel &lv = d->lv[l];
      if (!lv.set) return amgb_fail(c, AMGB_ESTATE, "layout of level %d missing", l);
      const int rows = lv.distributed ? lv.n_owned : lv.n_global;
      if (c->A[l].nrows != rows || c->A[l].ncols != lv.n_ext()) return amgb_fail(c, AMGB_EINVAL, "A_%d block shape does not match its layout", l);
      if (l < L - 1) {
         const DistLevel &nx = d->lv[l + 1];
         const int prow = rows, pcol = nx.n_ext();
         const int rrow = lv.distributed ? nx.n_owned : nx.n_global, rcol = lv.n_ext();
         if (c->P[l].nrows != prow || c->P[l].ncols != pcol || c->R[l].nrows != rrow || c->R[l].ncols != rcol)
            return amgb_fail(c, AMGB_EINVAL, "transfer block shapes at level %d do not match the layouts", l);
      }
   }
   d->ws.assign(L, nullptr); d->r.assign(L, nullptr); d->e.assign(L, nullptr);
   d->t.assign(L, nullptr); d->w.assign(L, nullptr);
   for (int l = 0; l < L; l++) {
      const DistLevel &lv = d->lv[l];
      const size_t bytes = sizeof(double) * (size_t)lv.n_ext();
      if ((rc = amgb_dev_alloc_bytes(c, (void **)&d->ws[l], bytes, true))) return rc;
      if ((rc = amgb_dev_alloc_bytes(c, (void **)&d->r[l], bytes, true))) return rc;
      if ((rc = amgb_dev_alloc_bytes(c, (void **)&d->e[l], bytes, true))) return rc;
      if (o.solver == AMGB_SOLVER_AFACX || mult) {
         if ((rc = amgb_dev_alloc_bytes(c, (void **)&d->t[l], bytes, true))) return rc;
         if ((rc = amgb_dev_alloc_bytes(c, (void **)&d->w[l], bytes, true))) return rc;
      }
      // w/d (1/l1 for L1-Jacobi; the row sums of a local row block are the global ones) of the owned rows, ghosts from the neighbours, then the column-scaled values of the one-pass
      // symmetrised smoother (on replicated levels amgb_setup already did this)
      CUDA_OK(c, cudaMemcpyAsync(d->ws[l] + lv.off(), l1s ? c->inv_l1[l] : c->ws[l], sizeof(double) * c->A[l].nrows, cudaMemcpyDeviceToDevice, c->stream));
      if (lv.distributed) {
         if ((rc = dist_halo(c, l, d->ws[l]))) return rc;
         if (c->A[l].va)      // (lean storage keeps no CSR copy of a sliced-ELL matrix)
            c->launches += launch_colscale(c->stream, c->A[l].nnz, c->A[l].ci, c->A[l].va, d->ws[l], const_cast<double *>(c->A[l].sval));
         if (c->A[l].sell_slices > 0)
            c->launches += launch_colscale(c->stream, (int)c->sell_entries[&c->A[l]], c->A[l].sell_ci, c->A[l].sell_va, d->ws[l],
                                           const_cast<double *>(c->A[l].sell_sval));
         if ((rc = amgb_build_sellu(c, c->A[l]))) return rc;      // (the scaled values of a partitioned level are final only now)
      }
   }
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&d->partials3, sizeof(double) * 3 * (size_t)c->npartials, true))) return rc;
   CUDA_OK(c, cudaStreamCreateWithFlags(&d->comm_stream, cudaStreamNonBlocking));
   CUDA_OK(c, cudaEventCreateWithFlags(&d->ev_x, cudaEventDisableTiming));
   CUDA_OK(c, cudaEventCreateWithFlags(&d->ev_h, cudaEventDisableTiming));
   if (const char *ov = getenv("AMGB_DIST_OVERLAP")) d->overlap = atoi(ov) != 0;
   d->use_graph = d->nranks == 1;
   if (const char *gv = getenv("AMGB_DIST_GRAPH")) d->use_graph = atoi(gv) != 0;
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&d->u, sizeof(double) * (size_t)d->lv[0].n_ext(), true))) return rc;
   if (c->opt.factor_level0) {
      if ((rc = amgb_dev_alloc_bytes(c, (void **)&d->t0, sizeof(double) * (size_t)d->lv[0].n_ext(), true))) return rc;
      if ((rc = amgb_dev_alloc_bytes(c, (void **)&d->v0, sizeof(double) * (size_t)d->lv[0].n_ext(), true))) return rc;
   }
   if ((rc = amgb_dev_alloc_bytes(c, (void **)&d->f, sizeof(double) * (size_t)std::max(1, c->A[0].nrows), true))) return rc;
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   d->halo_bytes = 0; d->collectives = 0;
   d->ready = true;
   return AMGB_OK;
#else
   return amgb_fail(c, AMGB_ENCCL, "library built without NCCL");
#endif
}

int amgb_dist_set_rhs(amgb_ctx *c, const double *f_owned)
{
   NEED_READY(c);
   if (!c->dist || !c->dist->ready) return amgb_fail(c, AMGB_ESTATE, "amgb_dist_setup not called");
   if (!f_owned) return amgb_fail(c, AMGB_EINVAL, "null rhs");
   CUDA_OK(c, cudaMemcpyAsync(c->dist->f, f_owned, sizeof(double) * c->A[0].nrows, cudaMemcpyHostToDevice, c->stream));
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   return AMGB_OK;
}

int amgb_dist_get_solution(amgb_ctx *c, double *u_owned)
{
   NEED_READY(c);
   if (!c->dist || !c->dist->ready) return amgb_fail(c, AMGB_ESTATE, "amgb_dist_setup not called");
   if (!u_owned) return amgb_fail(c, AMGB_EINVAL, "null buffer");
   CUDA_OK(c, cudaMemcpyAsync(u_owned, c->dist->u + c->dist->lv[0].off(), sizeof(double) * c->A[0].nrows, cudaMemcpyDeviceToHost, c->stream));
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   return AMGB_OK;
}

// DMEM_Add's loop (src/DMEM_Add.cpp:101-130) for the synchronous Multadd cycle: x0 = 0; cycle; residual;
// global norm; stop test -- the same on every rank (the norm is all-reduced), so all ranks leave together.
int amgb_dist_solve_sync(amgb_ctx *c, double tol, int max_cycles, double *hist, int *n_cycles, double *solve_seconds)
{
   return amgb_dist_solve_sync_accel(c, tol, max_cycles, 0, 1.0, 1.0, hist, n_cycles, solve_seconds);
}

// accel 1 / 2: DMEM_ChebyUpdate (src/DMEM_Misc.cpp:612-666) applied to the accumulated correction in
// DMEM_SyncAddCorrect (src/DMEM_Add.cpp:706-711): cycle 0: d = e; then d = (omega-1) d + omega*delta*e; x += d, with
// omega from the Chebyshev recurrence c_{k+1} = 2 mu c_k - c_{k-1} (accel 1) or fixed 2/(1+sqrt(1-mu^-2)) (accel 2).
int amgb_dist_solve_sync_accel(amgb_ctx *c, double tol, int max_cycles, int accel, double mu, double delta, double *hist,
                               int *n_cycles, double *solve_seconds)
{
   NEED_READY(c);
#ifdef AMG_HAVE_NCCL
   DistState *d = c->dist;
   if (!d || !d->ready) return amgb_fail(c, AMGB_ESTATE, "amgb_dist_setup not called");
   if (max_cycles < 0 || accel < 0 || accel > 2) return amgb_fail(c, AMGB_EINVAL, "bad arguments");
   const bool mult = c->opt.solver == AMGB_SOLVER_MULT;
   if (mult && accel)
      return amgb_fail(c, AMGB_EINVAL, "accel %d: DMEM_ChebyUpdate accelerates the additive correction, not the MULT V-cycle", accel);
   int rc;
   const int nown = c->A[0].nrows;
   double *uo = d->u + d->lv[0].off();
   if (accel && !d->ecyc) {
      if ((rc = amgb_dev_alloc_bytes(c, (void **)&d->ecyc, sizeof(double) * (size_t)std::max(1, nown), true))) return rc;
      if ((rc = amgb_dev_alloc_bytes(c, (void **)&d->dacc, sizeof(double) * (size_t)std::max(1, nown), true))) return rc;
   }
   double c_prev = 1.0, c_cur = mu;
   CUDA_OK(c, cudaMemsetAsync(d->u, 0, sizeof(double) * (size_t)d->lv[0].n_ext(), c->stream));
   if (mult)     // the level iterates of the V-cycle start from zero in every solve (the coarsest one carries over between cycles)
      for (int l = 1; l < c->L; l++) CUDA_OK(c, cudaMemsetAsync(d->e[l], 0, sizeof(double) * (size_t)d->lv[l].n_ext(), c->stream));
   if ((rc = dist_residual(c))) return rc;
   double ss;
   if ((rc = amgb_fetch_scalar(c, &ss))) return rc;
   const double r0 = sqrt(ss);
   if (hist) hist[0] = 1.0;
   int done = 0;
   // (the graph is captured only after ONE cycle has run with per-operation launches -- d->graph_warm: NCCL connects
   //  peers and algorithms lazily at first use (NCCL_RUNTIME_CONNECT), and the first all-gather of a solve would otherwise
   //  meet that set-up INSIDE the capture, where its host-side exchange and CUDA calls cannot run)
   if (d->use_graph && !accel && !d->graph_exec && d->graph_warm) {
      // capture u += B r; r = f - A u; ||r||^2 all-reduced; 8-byte D2H.  The halo exchanges run on the communication stream,
      // which joins the capture through the events dist_spmv records and is joined back before every boundary launch.
      cudaGraph_t g;
      const long long l0 = c->launches, h0 = d->halo_bytes, c0 = d->collectives;
      CUDA_OK(c, cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
      rc = dist_iteration(c);
      cudaMemcpyAsync(c->h_scalars, c->d_scalars, sizeof(double), cudaMemcpyDeviceToHost, c->stream);
      cudaError_t ce = cudaStreamEndCapture(c->stream, &g);
      if (rc) return rc;
      if (ce != cudaSuccess) return amgb_fail(c, AMGB_ECUDA, "graph capture of the partitioned cycle failed: %s", cudaGetErrorString(ce));
      d->graph_kernels = c->launches - l0; d->graph_halo_bytes = d->halo_bytes - h0; d->graph_collectives = d->collectives - c0;
      c->launches = l0; d->halo_bytes = h0; d->collectives = c0;
      CUDA_OK(c, cudaGraphInstantiate(&d->graph_exec, g, 0));
      cudaGraphDestroy(g);
   }
   CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
   for (int k = 1; k <= max_cycles; k++) {
      if (d->graph_exec && !accel) {
         CUDA_OK(c, cudaGraphLaunch(d->graph_exec, c->stream));
         {
            // a replay that never completes (collectives of two ranks that do not meet) must fail, not hang the job
            const double t_start = omp_get_wtime();
            cudaError_t q;
            while ((q = cudaStreamQuery(c->stream)) == cudaErrorNotReady)
               if (omp_get_wtime() - t_start > 60.0)
                  return amgb_fail(c, AMGB_ENCCL, "replay of the captured partitioned cycle did not complete within 60 s (cycle %d): "
                                                  "set AMGB_DIST_GRAPH=0", k);
            CUDA_OK(c, q);
         }
         c->launches += d->graph_kernels; d->halo_bytes += d->graph_halo_bytes; d->collectives += d->graph_collectives;
         ss = c->h_scalars[0];
         done = k;
         const double relg = sqrt(ss) / r0;
         if (hist) hist[k] = relg;
         if (relg < tol) break;
         continue;
      }
      if (!accel) {
         if ((rc = dist_iteration(c))) return rc;
      } else {
         if ((rc = dist_cycle(c, d->ecyc, false))) return rc;
         if (k == 1) c->launches += launch_axpby(c->cfg, c->stream, nown, 1.0, d->ecyc, 0.0, d->dacc, nullptr);
         else {
            double omega;
            if (accel == 2) omega = 2.0 / (1.0 + sqrt(1.0 - 1.0 / (mu * mu)));
            else {
               const double c_temp = c_cur;
               c_cur = 2.0 * mu * c_cur - c_prev;
               c_prev = c_temp;
               omega = 2.0 * mu * c_prev / c_cur;
            }
            c->launches += launch_axpby(c->cfg, c->stream, nown, omega * delta, d->ecyc, omega - 1.0, d->dacc, nullptr);
         }
         c->launches += launch_add(c->cfg, c->stream, nown, d->dacc, uo);
         if ((rc = dist_residual(c))) return rc;
      }
      if ((rc = amgb_fetch_scalar(c, &ss))) return rc;
      done = k;
      const double rel = sqrt(ss) / r0;
      if (hist) hist[k] = rel;
      if (rel < tol) break;
      if (d->use_graph && !accel && !d->graph_exec) {
         // every NCCL operation of a cycle has now run once outside a capture: capture the cycle for the remaining iterations
         d->graph_warm = true;
         cudaGraph_t g;
         const long long l0 = c->launches, h0 = d->halo_bytes, c0 = d->collectives;
         CUDA_OK(c, cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
         rc = dist_iteration(c);
         cudaMemcpyAsync(c->h_scalars, c->d_scalars, sizeof(double), cudaMemcpyDeviceToHost, c->stream);
         cudaError_t ce = cudaStreamEndCapture(c->stream, &g);
         if (rc) return rc;
         if (ce != cudaSuccess) return amgb_fail(c, AMGB_ECUDA, "graph capture of the partitioned cycle failed: %s", cudaGetErrorString(ce));
         d->graph_kernels = c->launches - l0; d->graph_halo_bytes = d->halo_bytes - h0; d->graph_collectives = d->collectives - c0;
         c->launches = l0; d->halo_bytes = h0; d->collectives = c0;
         CUDA_OK(c, cudaGraphInstantiate(&d->graph_exec, g, 0));
         cudaGraphDestroy(g);
      }
   }
   CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
   CUDA_OK(c, cudaEventSynchronize(c->ev1));
   float ms = 0;
   cudaEventElapsedTime(&ms, c->ev0, c->ev1);
   if (solve_seconds) *solve_seconds = ms * 1e-3;
   if (n_cycles) *n_cycles = done;
   c->r0_norm = r0;
   CUDA_OK(c, cudaGetLastError());
   return AMGB_OK;
#else
   (void)tol; (void)max_cycles; (void)accel; (void)mu; (void)delta; (void)hist; (void)n_cycles; (void)solve_seconds;
   return amgb_fail(c, AMGB_ENCCL, "library built without NCCL");
#endif
}

// ---- DMEM_PowerMult (src/DMEM_Eig.cpp:10-104): extreme eigenvalues of B*A by power iteration on the partitioned path ----
// Same iteration as EigsPower: normalise, f = A u, u = B f from a zero guess; eig_max = <v, BAv> after `iters` steps; a second pass
// deflated with u <- BAv - eig_max v gives eig_min; DMEM's ChebySetup then takes alpha = eig_min, beta = eig_max
// (src/DMEM_Setup.cpp:1901-1914).  B = the partitioned additive cycle of this context (the reference applies hypre's own
// BoomerAMGSolve there whatever -solver says -- un-vendored; for the additive solvers the bounds that matter are those of the
// cycle being accelerated).  u0_owned: this rank's rows of the start vector (the reference draws RandDouble(0,1) - .5 after
// srand(rank)); NULL = all ones (EigsPower's start vector).  Inner products are all-reduced: every rank gets the same bounds.
int amgb_dist_eigs_power(amgb_ctx *c, int iters, const double *u0_owned, double *eig_min, double *eig_max)
{
   NEED_READY(c);
#ifdef AMG_HAVE_NCCL
   DistState *d = c->dist;
   if (!d || !d->ready) return amgb_fail(c, AMGB_ESTATE, "amgb_dist_setup not called");
   if (iters < 1 || !eig_min || !eig_max) return amgb_fail(c, AMGB_EINVAL, "bad arguments");
   if (c->opt.solver == AMGB_SOLVER_MULT)
      return amgb_fail(c, AMGB_EINVAL, "DMEM_PowerMult applies the additive cycles: the MULT V-cycle has no zero-guess linear form here");
   int rc;
   const int nown = c->A[0].nrows, off0 = d->lv[0].off();
   if (!d->ecyc) {
      if ((rc = amgb_dev_alloc_bytes(c, (void **)&d->ecyc, sizeof(double) * (size_t)std::max(1, nown), true))) return rc;
      if ((rc = amgb_dev_alloc_bytes(c, (void **)&d->dacc, sizeof(double) * (size_t)std::max(1, nown), true))) return rc;
   }
   double *uo = d->u + off0, *y = d->ecyc;
   auto global_dot = [&](const double *a, const double *b, double *out) -> int {
      int grid = 0;
      c->launches += launch_dot(c->cfg, c->stream, nown, a, b, c->partials, &grid);
      c->launches += launch_reduce_partials(c->stream, c->partials, grid, c->d_scalars);
      NCCL_OK(c, ncclAllReduce(c->d_scalars, c->d_scalars, 1, ncclDouble, ncclSum, d->comm, c->stream));
      d->collectives++;
      return amgb_fetch_scalar(c, out);
   };
   std::vector<double> ones;
   if (!u0_owned) { ones.assign((size_t)std::max(1, nown), 1.0); u0_owned = ones.data(); }
   double lam[2] = {0.0, 0.0};
   for (int pass = 0; pass < 2; pass++) {
      CUDA_OK(c, cudaMemsetAsync(d->u, 0, sizeof(double) * (size_t)d->lv[0].n_ext(), c->stream));
      CUDA_OK(c, cudaMemcpyAsync(uo, u0_owned, sizeof(double) * (size_t)nown, cudaMemcpyHostToDevice, c->stream));
      CUDA_OK(c, cudaStreamSynchronize(c->stream));
      for (int it = 1;; it++) {
         double ss;
         if ((rc = global_dot(uo, uo, &ss))) return rc;
         c->launches += launch_axpby(c->cfg, c->stream, nown, 1.0 / sqrt(ss), uo, 0.0, uo, y);                      // u /= |u|; y = u
         if ((rc = dist_spmv(c, c->A[0], false, 0, d->u, d->r[0] + off0, epi(1.0, 0.0, nullptr), false))) return rc;   // f = A u
         if ((rc = dist_cycle(c, uo, false))) return rc;                                                               // u = B f
         if (it == iters) break;
         if (pass == 1) c->launches += launch_axpby(c->cfg, c->stream, nown, -lam[0], y, 1.0, uo, nullptr);
      }
      if ((rc = global_dot(y, uo, &lam[pass]))) return rc;
   }
   *eig_max = lam[0];
   *eig_min = lam[1];
   CUDA_OK(c, cudaGetLastError());
   return AMGB_OK;
#else
   (void)iters; (void)u0_owned; (void)eig_min; (void)eig_max;
   return amgb_fail(c, AMGB_ENCCL, "library built without NCCL");
#endif
}

// ---- asynchronous fine-grid smoother across GPUs --------------------------------------------------------------------
// DMEM_AsyncSmooth (src/DMEM_Smooth.cpp:16-313; solver option of DMEM_Add, src/DMEM_Add.cpp:88-95) with the ASYNC_JACOBI /
// ASYNC_L1_JACOBI smoothers: every rank relaxes its rows of the fine system over and over, u = r ./ s, x += u, and ships
// the new boundary values to its neighbours without ever waiting for theirs -- it simply uses whatever ghost values have
// arrived (the reference keeps the residual incrementally, r -= A_diag e, r -= A_offd x_ghost as messages land,
// :226-262; that is r = b - A [x_own | x_ghost] with the ghosts of the moment).  The reference's MPI_Isend / Test engine
// (DMEM_Comm.cpp:81-382, finestIntra_outsideSend / Recv) becomes plain stores over NVLink: the neighbours' solution
// vectors are mapped through CUDA IPC and this rank writes its boundary entries straight into their ghost slots.
// Stop rule: the reference's LOCAL one -- every rank stops after `sweeps` own relaxations (AsyncSmoothCheckConverge :340-349).
int amgb_dist_ipc_export_solution(amgb_ctx *c, unsigned char handle64[64])
{
   NEED_READY(c);
   if (!c->dist || !c->dist->ready) return amgb_fail(c, AMGB_ESTATE, "amgb_dist_setup not called");
   cudaIpcMemHandle_t h;
   CUDA_OK(c, cudaIpcGetMemHandle(&h, c->dist->u));
   memcpy(handle64, &h, 64);
   return AMGB_OK;
}

// handle_lo / handle_hi: the exported handles of rank-1 / rank+1 (NULL at the ends of the chain, or for a neighbour that
// lives in this very process); lo_ghost_offset = index of rank-1's first ghost_hi entry in ITS level-0 vector
// (its halo_lo + its n_owned).  rank+1's ghost_lo entries start at index 0 of its vector.
int amgb_dist_ipc_open_neighbours(amgb_ctx *c, const unsigned char *handle_lo, long long lo_ghost_offset, const unsigned char *handle_hi)
{
   NEED_READY(c);
   DistState *d = c->dist;
   if (!d || !d->ready) return amgb_fail(c, AMGB_ESTATE, "amgb_dist_setup not called");
   if (d->nbr_lo || d->nbr_hi) return amgb_fail(c, AMGB_ESTATE, "neighbours already mapped");
   if ((handle_lo && d->rank == 0) || (handle_hi && d->rank == d->nranks - 1) || lo_ghost_offset < 0)
      return amgb_fail(c, AMGB_EINVAL, "no such neighbour");
   cudaIpcMemHandle_t h;
   void *ptr = nullptr;
   if (handle_lo) {
      memcpy(&h, handle_lo, 64);
      CUDA_OK(c, cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
      d->nbr_lo = (double *)ptr;
      d->nbr_lo_off = (long)lo_ghost_offset;
   }
   if (handle_hi) {
      memcpy(&h, handle_hi, 64);
      CUDA_OK(c, cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
      d->nbr_hi = (double *)ptr;
   }
   return AMGB_OK;
}

// `sweeps` relaxations of this rank's rows of A_0 x = f from the resident x (amgb_dist_solve_sync leaves its solution there;
// amgb_dist_set_rhs + a fresh context start from x = 0), enqueued on the context's stream; returns without waiting for
// the GPU.  Every sweep: x_own <- x_own + s o (f - A_0 [ghost_lo | x_own | ghost_hi]), then the boundary entries go to
// the neighbours' ghost slots.  With one rank this is `sweeps` sweeps of (L1-)Jacobi.
int amgb_dist_async_smooth(amgb_ctx *c, int sweeps)
{
   NEED_READY(c);
   DistState *d = c->dist;
   if (!d || !d->ready) return amgb_fail(c, AMGB_ESTATE, "amgb_dist_setup not called");
   if (sweeps < 0) return amgb_fail(c, AMGB_EINVAL, "sweeps < 0");
   const DistLevel &L0 = d->lv[0];
   if (L0.distributed && ((d->rank > 0 && L0.send_lo && !d->nbr_lo) || (d->rank < d->nranks - 1 && L0.send_hi && !d->nbr_hi)))
      return amgb_fail(c, AMGB_ESTATE, "amgb_dist_ipc_open_neighbours not called");
   const int nown = c->A[0].nrows;
   int rc;
   if (!d->sm_scratch && (rc = amgb_dev_alloc_bytes(c, (void **)&d->sm_scratch, sizeof(double) * (size_t)std::max(1, nown), true))) return rc;
   double *uo = d->u + L0.off();
   const double *so = d->ws[0] + L0.off();
   for (int k = 0; k < sweeps; k++) {
      enq_spmv(c, c->A[0], false, d->u, d->sm_scratch, epi(-1.0, 1.0, d->f, 1.0, uo, so), false);
      CUDA_OK(c, cudaMemcpyAsync(uo, d->sm_scratch, sizeof(double) * (size_t)nown, cudaMemcpyDeviceToDevice, c->stream));
      if (d->nbr_lo && L0.send_lo)
         CUDA_OK(c, cudaMemcpyAsync(d->nbr_lo + d->nbr_lo_off, uo, sizeof(double) * (size_t)L0.send_lo, cudaMemcpyDefault, c->stream));
      if (d->nbr_hi && L0.send_hi)
         CUDA_OK(c, cudaMemcpyAsync(d->nbr_hi, uo + L0.n_owned - L0.send_hi, sizeof(double) * (size_t)L0.send_hi, cudaMemcpyDefault, c->stream));
      d->halo_bytes += 8LL * ((d->nbr_lo ? L0.send_lo : 0) + (d->nbr_hi ? L0.send_hi : 0));
   }
   CUDA_OK(c, cudaGetLastError());
   return AMGB_OK;
}

// global ||f - A_0 x||_2 of the resident vectors: a synchronised halo exchange, the residual and an all-reduce (collective)
int amgb_dist_residual_norm(amgb_ctx *c, double *norm)
{
   NEED_READY(c);
#ifdef AMG_HAVE_NCCL
   DistState *d = c->dist;
   if (!d || !d->ready) return amgb_fail(c, AMGB_ESTATE, "amgb_dist_setup not called");
   if (!norm) return amgb_fail(c, AMGB_EINVAL, "null output");
   int rc;
   if ((rc = dist_residual(c))) return rc;
   double ss;
   if ((rc = amgb_fetch_scalar(c, &ss))) return rc;
   *norm = sqrt(ss);
   return AMGB_OK;
#else
   (void)norm;
   return amgb_fail(c, AMGB_ENCCL, "library built without NCCL");
#endif
}

int amgb_dist_zero_solution(amgb_ctx *c)
{
   NEED_READY(c);
   if (!c->dist || !c->dist->ready) return amgb_fail(c, AMGB_ESTATE, "amgb_dist_setup not called");
   CUDA_OK(c, cudaMemsetAsync(c->dist->u, 0, sizeof(double) * (size_t)c->dist->lv[0].n_ext(), c->stream));
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   return AMGB_OK;
}

// halo bytes sent and NCCL operations enqueued by this rank since amgb_dist_setup
int amgb_dist_stats(amgb_ctx *c, long long *halo_bytes, long long *collectives)
{
   if (!c || !c->dist) return AMGB_EINVAL;
   if (halo_bytes) *halo_bytes = c->dist->halo_bytes;
   if (collectives) *collectives = c->dist->collectives;
   return AMGB_OK;
}

}   // extern "C"

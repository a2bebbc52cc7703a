// ctx.h -- internal context shared by context.cu / async.cu / dist.cu (not part of the C ABI).
#pragma once
#include "amg_b200.h"
#include "launch.h"
#include <map>
#include <vector>

struct DistState;
struct ExtState;

struct amgb_ctx {
   int device = 0;
   cudaStream_t stream = nullptr;
   cudaEvent_t ev0 = nullptr, ev1 = nullptr;
   LaunchCfg cfg;
   amgb_options opt;
   int L = 0;
   bool ready = false;
   bool symmetric = false;
   std::vector<DevCSR> A, P, R;
   std::vector<int *> jgs_bounds;   // per level: explicit Gauss-Seidel block list of the hybrid smoother (device, nb + 1 ints) or null
   std::vector<int> jgs_nb;
   DevCSR Ainv;                     // dense inverse of the coarsest operator (coarse_solve), stored as a full CSR
   std::vector<int> hA;
   std::map<const DevCSR *, long> sell_entries;
   std::vector<int> last_perm;      // host copies of the last built SELL permutation / block list (unit classification)
   std::vector<int4> last_blk;
   // per level: w/d, d/w, l1, 1/l1; residual chain, correction chain, two scratch vectors
   std::vector<double *> ws, dow, l1, inv_l1, r, e, t, w;
   double *f = nullptr, *u = nullptr, *cvec = nullptr, *u_outer = nullptr, *y_outer = nullptr;
   double *io_a = nullptr, *io_b = nullptr, *io_c = nullptr;
   int io_len = 0;                  // entries of the three staging vectors (largest row / column count of the hierarchy)
   std::vector<double *> lean_diag, lean_l1;   // lean storage: diagonal and l1 norms of A_l formed on the host at upload
   double *partials = nullptr;
   int npartials = 0;
   double *d_scalars = nullptr;
   double *h_scalars = nullptr;   // pinned
   double r0_norm = 0.0;
   cudaGraphExec_t graph_exec = nullptr;
   long long graph_kernels = 0;
   // preconditioned conjugate gradients (pcg.cu): direction p, A p, the device scalars (PCG_* slots), one iteration's graph
   double *pcg_p = nullptr, *pcg_q = nullptr, *pcg_s = nullptr;
   cudaGraphExec_t pcg_graph = nullptr;
   long long pcg_graph_kernels = 0;
   long long launches = 0;
   size_t bytes_allocated = 0;
   int host_threads = 1;   // threads for the upload-time layout conversions (set in amgb_create)
   long sellu_slices = 0, sellu_groups = 0;               // SELL-U: encoded slices / groups over the whole hierarchy
   size_t l2_bytes = 0, max_window = 0, persist_max = 0;
   std::vector<void *> allocs;
   // async
   void *async_params_dev = nullptr;
   AsyncParams *async_host = nullptr;
   // one contiguous arena for the coarse hierarchy, so that ONE access-policy window can pin it in L2 for the
   // persistent asynchronous kernel (every level group re-reads it once per correction)
   char *arena = nullptr;
   size_t arena_size = 0, arena_used = 0;
   bool alloc_in_arena = false;
   cudaAccessPolicyWindow window = {};
   bool window_valid = false;
   bool async_ready = false, async_balanced = false, async_heavy = false;
   int async_grid = 0, async_grid_used = 0, async_first = 0;
   std::vector<int> async_cta_begin;
   std::vector<double> async_work;          // cost model of every group's program (seeds the CTA groups)
   std::vector<double *> async_vec;         // [group][vector kind][level] -> device pointer of a group-private vector
   double *async_r_shared = nullptr;        // shared residual (-res_compute_type global / -read_type res)
   // distributed
   DistState *dist = nullptr;
   // implicit extended-system BPX solver: per-level vectors (extended.cu)
   ExtState *ext = nullptr;
   // asynchronous solve across GPUs: IPC-mapped solution vectors of the peer ranks (fp64 reductions over NVLink)
   std::vector<double *> peer_u;
   char err[512] = {0};
};

int amgb_fail(amgb_ctx *c, int code, const char *fmt, ...);
// owned column range [c0, c1) of the input vector of matrix (kind, level) on a partitioned level; false if the
// input vector is not partitioned (nothing to overlap)
bool amgb_dist_owned_cols(const amgb_ctx *c, int kind, int level, int *c0, int *c1);
void amgb_dist_teardown(amgb_ctx *c);
void amgb_ext_teardown(amgb_ctx *c);
void amgb_pcg_teardown(amgb_ctx *c);      // frees the conjugate-gradient vectors and graph
void amgb_async_teardown(amgb_ctx *c);   // frees the host copy of the persistent kernel's parameter block
// persistent kernel, host side (async.cu), shared with the row-partitioned solve (dist_async.cu)
double async_op_cost(const DevCSR &M, long sell_entries);                      // cost-model seed of the CTA groups
void async_assign_groups(amgb_ctx *c, const std::vector<double> &work);        // CTA groups in proportion to `work`
int amgb_dist_diag_offset(const amgb_ctx *c, int level);          // position of the diagonal in a local row block
bool amgb_dist_level_distributed(const amgb_ctx *c, int level);

#define CUDA_OK(c, call)                                                                                   \
   do {                                                                                                    \
      cudaError_t e__ = (call);                                                                            \
      if (e__ != cudaSuccess)                                                                              \
         return amgb_fail((c), AMGB_ECUDA, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(e__)); \
   } while (0)

#define NEED_READY(c)                                                                      \
   do {                                                                                    \
      if (!(c)) return AMGB_EINVAL;                                                        \
      if (!(c)->ready) return amgb_fail((c), AMGB_ESTATE, "amgb_setup not called");        \
      CUDA_OK((c), cudaSetDevice((c)->device));                                            \
   } while (0)

// helpers exported by context.cu to async.cu / dist.cu
int amgb_dev_alloc_bytes(amgb_ctx *c, void **p, size_t bytes, bool zero);
int amgb_build_sellu(amgb_ctx *c, DevCSR &M);   // SELL-U encoding of a sliced-ELL matrix whose scaled values are final
void enq_spmv(amgb_ctx *c, const DevCSR &M, bool sval, const double *x, double *y, const SpmvEpilogue &e, bool norm);
void enq_residual(amgb_ctx *c);
void enq_spmv_dot(amgb_ctx *c, const DevCSR &M, bool sval, const double *x, double *y, const SpmvEpilogue &e, const double *w, double *dot_out);
void enq_cycle(amgb_ctx *c, double *target, bool accumulate, const double *dot_w = nullptr, double *dot_out = nullptr);
int amgb_fetch_scalar(amgb_ctx *c, double *out);

// context.cu -- C ABI (include/amg_b200.h): context, hierarchy upload, per-op entry points,
// synchronous cycles (Multadd / AFACx / BPX) and the outer solve loop, all enqueued on one CUDA
// stream and replayed as a CUDA graph per iteration.
//
// Reference call paths replaced (host orchestration only; the arithmetic lives in kernels.cu):
//   SMEM_Solve sync branch          src/SMEM_Solve.cpp:93-252
//   SMEM_Sync_Add_Vcycle            src/SMEM_Sync_AMG.cpp:408-621  (meaning: src/SEQ_AMG.cpp:110-235)
//   SMEM_Sync_Parfor_BPXcycle       src/SMEM_Sync_AMG.cpp:147-294
//   SMEM_Sync_Parfor_AFACx_Vcycle   src/SMEM_Sync_AMG.cpp:296-406
//   SMEM_Smooth dispatcher          src/SMEM_Solve.cpp:264-377
#include "ctx.h"
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>
#include <omp.h>

int amgb_fail(amgb_ctx *c, int code, const char *fmt, ...)
{
   if (c) {
      va_list ap;
      va_start(ap, fmt);
      vsnprintf(c->err, sizeof(c->err), fmt, ap);
      va_end(ap);
   }
   return code;
}

// ---- device memory helpers ----------------------------------------------------------------------
template <class T>
static int dev_alloc(amgb_ctx *c, T **p, size_t n)
{
   *p = nullptr;
   n += 64 / sizeof(T) + 8;   // slack: 16-byte granular bulk copies may touch a few elements past the end
   if (c->alloc_in_arena && c->arena) {
      const size_t bytes = (n * sizeof(T) + 255) & ~(size_t)255;
      if (c->arena_used + bytes <= c->arena_size) {
         *p = reinterpret_cast<T *>(c->arena + c->arena_used);
         c->arena_used += bytes;
         return AMGB_OK;
      }
   }
   cudaError_t e = cudaMalloc((void **)p, n * sizeof(T));
   if (e != cudaSuccess) return amgb_fail(c, AMGB_ENOMEM, "cudaMalloc(%zu bytes): %s", n * sizeof(T), cudaGetErrorString(e));
   c->allocs.push_back((void *)*p);
   c->bytes_allocated += n * sizeof(T);
   return AMGB_OK;
}
template <class T>
static int dev_upload(amgb_ctx *c, T **p, const T *h, size_t n)
{
   int rc = dev_alloc(c, p, n);
   if (rc) return rc;
   if (n) CUDA_OK(c, cudaMemcpyAsync(*p, h, n * sizeof(T), cudaMemcpyHostToDevice, c->stream));
   return AMGB_OK;
}
static int dev_zero(amgb_ctx *c, double **p, size_t n)
{
   int rc = dev_alloc(c, p, n);
   if (rc) return rc;
   CUDA_OK(c, cudaMemsetAsync(*p, 0, std::max<size_t>(n, 1) * sizeof(double), c->stream));
   return AMGB_OK;
}

int amgb_dev_alloc_bytes(amgb_ctx *c, void **p, size_t bytes, bool zero)
{
   char *q = nullptr;
   int rc = dev_alloc(c, &q, bytes);
   if (rc) return rc;
   if (zero) CUDA_OK(c, cudaMemsetAsync(q, 0, std::max<size_t>(bytes, 1), c->stream));
   *p = q;
   return AMGB_OK;
}

extern "C" {

void amgb_default_options(amgb_options *o)
{
   // src/SMEM_Main.cpp:64-104
   o->solver = AMGB_SOLVER_MULTADD;
   o->smoother = AMGB_SMOOTH_JACOBI;
   o->smooth_weight = 1.0;
   o->num_pre_smooth_sweeps = 1;
   o->num_post_smooth_sweeps = 1;
   o->num_fine_smooth_sweeps = 1;
   o->num_coarse_smooth_sweeps = 1;
   o->jgs_block_rows = 8;
   o->use_sell = 1;
   o->l2_persist = 1;
   o->use_stream = 1;
   o->factor_level0 = 0;
   o->coarse_solve = 0;
   o->stream_variant = 8;
   o->sell_sigma = 128;
   o->sell_uniform = 1;
   o->async_type = 0;
   o->res_compute_type = 0;
   o->read_type = 0;
   o->lean_storage = 0;
   o->factor_restriction = 0;
   o->sell_window_epilogue = 1;
}

int amgb_create(amgb_ctx **out, int device)
{
   if (!out) return AMGB_EINVAL;
   *out = nullptr;
   int ndev = 0;
   cudaError_t e = cudaGetDeviceCount(&ndev);
   if (e != cudaSuccess || ndev == 0) return AMGB_ECUDA;   // no CPU fallback by design
   if (device < 0 || device >= ndev) return AMGB_EINVAL;
   amgb_ctx *c = new amgb_ctx();
   c->device = device;
   if (cudaSetDevice(device) != cudaSuccess) { delete c; return AMGB_ECUDA; }
   cudaDeviceProp prop;
   cudaGetDeviceProperties(&prop, device);
   c->cfg.num_sms = prop.multiProcessorCount;
   c->cfg.ctas_per_sm = 8;
   c->host_threads = std::max(1, std::min(16, omp_get_num_procs()));
   c->l2_bytes = prop.l2CacheSize;
   c->max_window = prop.accessPolicyMaxWindowSize;
   c->persist_max = prop.persistingL2CacheMaxSize;
   if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return AMGB_ECUDA; }
   // L2 persistence for the coarse hierarchy: at most half of what the device lets us set aside
   if (c->persist_max > 0 && c->max_window > 0) {
      const size_t want = std::min<size_t>(std::min(c->persist_max, c->max_window), (size_t)48 << 20);
      if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want) == cudaSuccess && cudaMalloc((void **)&c->arena, want) == cudaSuccess) {
         c->arena_size = want;
         c->allocs.push_back(c->arena);
      } else {
         c->arena = nullptr;
         cudaGetLastError();
      }
   }
   cudaEventCreate(&c->ev0);
   cudaEventCreate(&c->ev1);
   cudaMallocHost((void **)&c->h_scalars, 64 * sizeof(double));
   amgb_default_options(&c->opt);
   c->cfg.sell_window_sigma = c->opt.sell_window_epilogue ? c->opt.sell_sigma : 0;
   *out = c;
   return AMGB_OK;
}

int amgb_destroy(amgb_ctx *c)
{
   if (!c) return AMGB_EINVAL;
   cudaSetDevice(c->device);
   cudaStreamSynchronize(c->stream);
   amgb_dist_teardown(c);
   for (double *p : c->peer_u) cudaIpcCloseMemHandle(p);
   amgb_async_teardown(c);
   amgb_ext_teardown(c);
   amgb_pcg_teardown(c);
   if (c->graph_exec) cudaGraphExecDestroy(c->graph_exec);
   for (void *p : c->allocs) cudaFree(p);
   if (c->h_scalars) cudaFreeHost(c->h_scalars);
   cudaEventDestroy(c->ev0);
   cudaEventDestroy(c->ev1);
   cudaStreamDestroy(c->stream);
   delete c;
   return AMGB_OK;
}

const char *amgb_last_error(const amgb_ctx *c) { return c ? c->err : "null context"; }
long long amgb_launch_count(const amgb_ctx *c) { return c ? c->launches : 0; }

int amgb_set_num_levels(amgb_ctx *c, int L)
{
   if (!c || L < 1 || L > AMGB_MAX_LEVELS) return amgb_fail(c, AMGB_EINVAL, "num_levels %d out of range", L);
   if (c->L) return amgb_fail(c, AMGB_ESTATE, "hierarchy already defined");
   c->L = L;
   c->A.resize(L); c->P.resize(L); c->R.resize(L);
   c->hA.resize(L);
   c->lean_diag.assign(L, nullptr); c->lean_l1.assign(L, nullptr);
   c->jgs_bounds.assign(L, nullptr); c->jgs_nb.assign(L, 0);
   return AMGB_OK;
}

int amgb_set_options(amgb_ctx *c, const amgb_options *o)
{
   if (!c || !o) return AMGB_EINVAL;
   if (o->smooth_weight == 0.0 || o->jgs_block_rows < 1) return amgb_fail(c, AMGB_EINVAL, "bad options");
   if (o->stream_variant != 8)
      return amgb_fail(c, AMGB_EINVAL, "stream_variant %d: the field is retired, only 8 (the warp-stream kernel) is accepted", o->stream_variant);
   if (c->L) return amgb_fail(c, AMGB_ESTATE, "amgb_set_options must precede the hierarchy upload");
   c->opt = *o;
   c->cfg.sell_window_sigma = o->sell_window_epilogue ? o->sell_sigma : 0;
   return AMGB_OK;
}

// choose lanes per row for the CSR vector kernel from the mean row length
static int pick_lpr(int nrows, int nnz)
{
   double avg = nrows > 0 ? (double)nnz / nrows : 0.0;
   if (avg <= 2.5) return 2;
   if (avg <= 5.0) return 4;
   if (avg <= 12.0) return 8;
   if (avg <= 28.0) return 16;
   return 32;
}

// Build the sliced-ELL (C = 32) copy on the host.  sigma == 1: rows in natural order, accepted when padding
// <= 15 % (stencil levels).  sigma > 1 (SELL-C-sigma): inside every window of `sigma` consecutive rows the rows are
// ordered by decreasing length before being cut into slices (sell_perm records slot -> row), which brings the
// padding of the Galerkin / transfer operators from 35-58 % down to ~11-15 % (sigma = 128) while the 32 rows of
// a slice stay within 128 rows of each other, so that one gather instruction still touches few lines of x.
static int build_sell(amgb_ctx *c, DevCSR &M, int nrows, const int *rp, const int *ci, const double *va, int sigma,
                      double max_padding)
{
   const int slices = (nrows + 31) / 32;
   std::vector<int> perm;
   if (sigma > 1) {
      perm.resize((size_t)slices * 32, -1);
      for (int r = 0; r < nrows; r++) perm[r] = r;
#pragma omp parallel for schedule(static)
      for (int w0 = 0; w0 < nrows; w0 += sigma) {
         const int w1 = std::min(nrows, w0 + sigma);
         std::stable_sort(perm.begin() + w0, perm.begin() + w1,
                          [&](int a, int b) { return rp[a + 1] - rp[a] > rp[b + 1] - rp[b]; });
      }
   }
   auto row_of = [&](int slot) { return sigma > 1 ? perm[slot] : (slot < nrows ? slot : -1); };
   std::vector<int> off((size_t)slices + 1, 0);
   long padded = 0;
   for (int s = 0; s < slices; s++) {
      int w = 0;
      for (int l = 0; l < 32; l++) {
         const int r = row_of(s * 32 + l);
         if (r >= 0) w = std::max(w, rp[r + 1] - rp[r]);
      }
      padded += (long)w * 32;
      if (padded > 2147483000L) return AMGB_OK;   // keep CSR
      off[s + 1] = (int)padded;
   }
   const long nnz = rp[nrows];
   if (nnz == 0 || (double)padded > (1.0 + max_padding) * (double)nnz) return AMGB_OK;
   std::vector<int> sci((size_t)padded);
   std::vector<double> sva((size_t)padded, 0.0);
#pragma omp parallel for schedule(static)
   for (int s = 0; s < slices; s++) {
      const int w = (off[s + 1] - off[s]) / 32;
      for (int l = 0; l < 32; l++) {
         const int r = row_of(s * 32 + l);
         for (int k = 0; k < w; k++) {
            const size_t d = (size_t)off[s] + (size_t)k * 32 + l;
            if (r >= 0 && rp[r] + k < rp[r + 1]) { sci[d] = ci[rp[r] + k]; sva[d] = va[rp[r] + k]; }
            else { sci[d] = (r >= 0 && rp[r + 1] > rp[r]) ? ci[rp[r]] : 0; sva[d] = 0.0; }   // padding: harmless gather, zero value
         }
      }
   }
   int *d_off, *d_ci; double *d_va;
   int rc;
   if ((rc = dev_upload(c, &d_off, off.data(), off.size()))) return rc;
   if ((rc = dev_upload(c, &d_ci, sci.data(), sci.size()))) return rc;
   if ((rc = dev_upload(c, &d_va, sva.data(), sva.size()))) return rc;
   c->last_perm = perm;
   if (sigma > 1) {
      int *d_perm;
      if ((rc = dev_upload(c, &d_perm, perm.data(), perm.size()))) return rc;
      M.sell_perm = d_perm;
   }
   CUDA_OK(c, cudaStreamSynchronize(c->stream));   // host vectors go out of scope
   M.sell_slices = slices; M.sell_off = d_off; M.sell_ci = d_ci; M.sell_va = d_va;
   c->sell_entries[&M] = padded;
   return AMGB_OK;
}

// SELL-U: re-encode the slices of a sigma = 1 sliced-ELL matrix whose entries take few distinct (column - row, value,
// scaled value) triples (see DevCSR::su_desc).  Runs at setup time, after the column-scaled values exist, on host copies of
// the device arrays (chunks of slices, OpenMP over slices).  Lossless: a slice is encoded only if every real entry of its
// rows falls into a group and no row holds the same column twice; a row's terms are then summed in group order (the order
// of first appearance in the slice) instead of CSR order.  A slice that would need more than half the bytes of its
// regular encoding keeps the regular one; a matrix where fewer than half of the slices qualify is left alone.
struct SuGrp { int delta; unsigned mask; double va, sv; };

// encode slices [s0, s1): ci / va / sv hold the sliced-ELL entries starting at entry offset e0 (= off[s0] for a chunk)
static void sellu_encode_chunk(int nrows, const int *off, const int *rp, int s0, int s1, size_t e0, const int *ci,
                               const double *va, const double *sv, std::vector<std::vector<SuGrp>> &gs)
{
   gs.assign((size_t)(s1 - s0), std::vector<SuGrp>());
#pragma omp parallel for schedule(dynamic, 1024)
   for (int s = s0; s < s1; s++) {
      const int w = (off[s + 1] - off[s]) / 32;
      if (w == 0) continue;
      std::vector<SuGrp> &g = gs[(size_t)(s - s0)];
      const size_t cap = std::min<size_t>(64, (size_t)w * 32 * 12 / 2 / 24);
      bool ok = true;
      for (int l = 0; l < 32 && ok; l++) {
         const int r = s * 32 + l;
         if (r >= nrows) break;
         const int len = rp[r + 1] - rp[r];
         for (int k = 0; k < len && ok; k++) {
            const size_t d = (size_t)off[s] - e0 + (size_t)k * 32 + l;
            const int delta = ci[d] - r;
            // the same column twice in ONE row is not representable (one mask bit per lane and group; two groups with
            // the same delta would be, but such a row is malformed anyway): leave the slice alone
            for (size_t q2 = 0; q2 < g.size(); q2++)
               if (g[q2].delta == delta && ((g[q2].mask >> l) & 1u)) { ok = false; break; }
            if (!ok) break;
            size_t q = 0;
            for (; q < g.size(); q++)
               if (g[q].delta == delta && memcmp(&g[q].va, &va[d], 8) == 0 && memcmp(&g[q].sv, &sv[d], 8) == 0) break;
            if (q == g.size()) {
               if (g.size() >= cap) { ok = false; break; }
               g.push_back(SuGrp{delta, 0u, va[d], sv[d]});
            }
            g[q].mask |= 1u << l;
         }
      }
      if (!ok) g.clear();
   }
}

// group lists of many slices are identical (a constant-coefficient stencil has one list per boundary pattern): the table
// keeps one copy of every distinct list, slice s points at it through desc[s] = {first group, count}
struct SuTable {
   std::vector<SuGrp> groups;
   std::map<std::string, int> seen;
   int2 add(const std::vector<SuGrp> &g)
   {
      if (g.empty()) return make_int2(0, 0);
      std::string key(reinterpret_cast<const char *>(g.data()), g.size() * sizeof(SuGrp));
      auto it = seen.find(key);
      if (it != seen.end()) return make_int2(it->second, (int)g.size());
      const int first = (int)groups.size();
      groups.insert(groups.end(), g.begin(), g.end());
      seen.emplace(std::move(key), first);
      return make_int2(first, (int)g.size());
   }
};

static int build_sellu(amgb_ctx *c, DevCSR &M)
{
   if (!c->opt.use_sell || c->opt.sell_uniform == 0 || M.sell_slices == 0 || M.sell_perm || M.su_desc || !M.sell_sval) return AMGB_OK;
   const int slices = M.sell_slices, nrows = M.nrows;
   std::vector<int> off((size_t)slices + 1), rp((size_t)nrows + 1);
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   CUDA_OK(c, cudaMemcpy(off.data(), M.sell_off, sizeof(int) * off.size(), cudaMemcpyDeviceToHost));
   CUDA_OK(c, cudaMemcpy(rp.data(), M.rp, sizeof(int) * rp.size(), cudaMemcpyDeviceToHost));
   std::vector<int2> desc((size_t)slices, make_int2(0, 0));
   const int CH = 262144;                                   // slices per chunk (bounds the host copy)
   SuTable tab;
   long encoded = 0, listed = 0;
   std::vector<int> ci;
   std::vector<double> va, sv;
   std::vector<std::vector<SuGrp>> gs;
   for (int s0 = 0; s0 < slices; s0 += CH) {
      const int s1 = std::min(slices, s0 + CH);
      const size_t e0 = (size_t)off[s0], ne = (size_t)off[s1] - e0;
      ci.resize(ne); va.resize(ne); sv.resize(ne);
      if (ne) {
         CUDA_OK(c, cudaMemcpy(ci.data(), M.sell_ci + e0, sizeof(int) * ne, cudaMemcpyDeviceToHost));
         CUDA_OK(c, cudaMemcpy(va.data(), M.sell_va + e0, sizeof(double) * ne, cudaMemcpyDeviceToHost));
         CUDA_OK(c, cudaMemcpy(sv.data(), M.sell_sval + e0, sizeof(double) * ne, cudaMemcpyDeviceToHost));
      }
      sellu_encode_chunk(nrows, off.data(), rp.data(), s0, s1, e0, ci.data(), va.data(), sv.data(), gs);
      for (int s = s0; s < s1; s++) {
         const std::vector<SuGrp> &g = gs[(size_t)(s - s0)];
         desc[s] = tab.add(g);
         if (!g.empty()) { encoded++; listed += (long)g.size(); }
      }
      // a matrix whose lists do not repeat (variable coefficients) would only trade one stream for another: give up early
      if (s1 >= std::min(slices, 65536) && (double)tab.groups.size() > 0.5 * (double)listed && tab.groups.size() > 4096) return AMGB_OK;
   }
   if (encoded * 2 < slices) return AMGB_OK;
   const std::vector<SuGrp> &all = tab.groups;
   std::vector<int2> dm(all.size());
   std::vector<double> gva(all.size()), gsv(all.size());
   for (size_t i = 0; i < all.size(); i++) { dm[i] = make_int2(all[i].delta, (int)all[i].mask); gva[i] = all[i].va; gsv[i] = all[i].sv; }
   int2 *d_desc, *d_dm; double *d_va, *d_sv;
   int rc;
   if ((rc = dev_upload(c, &d_desc, desc.data(), desc.size()))) return rc;
   if ((rc = dev_upload(c, &d_dm, dm.data(), dm.size()))) return rc;
   if ((rc = dev_upload(c, &d_va, gva.data(), gva.size()))) return rc;
   if ((rc = dev_upload(c, &d_sv, gsv.data(), gsv.size()))) return rc;
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   M.su_desc = d_desc; M.su_dm = d_dm; M.su_va = d_va; M.su_sval = d_sv;
   c->sellu_slices += encoded;
   c->sellu_groups += (long)all.size();
   return AMGB_OK;
}

// Host-only probe of the SELL-U encoder for the CPU test suite (no CUDA call): CSR + scaled values in, the sigma = 1 sliced-ELL
// layout is formed as build_sell does, encoded and deduplicated exactly as build_sellu does; out: per slice the first group
// and the group count (two ints per slice, count 0 = not encoded) and per group of the deduplicated table delta / mask / va / sv
// (malloc'ed, release with amgb_host_free).  Returns the number of slices.
int amgb_sellu_encode_host(int nrows, const int *rp, const int *ci, const double *va, const double *sv, int **desc_out,
                           int **delta_out, unsigned int **mask_out, double **gva_out, double **gsv_out, int *ngroups)
{
   const int slices = (nrows + 31) / 32;
   std::vector<int> off((size_t)slices + 1, 0);
   for (int s = 0; s < slices; s++) {
      int w = 0;
      for (int l = 0; l < 32 && s * 32 + l < nrows; l++) w = std::max(w, rp[s * 32 + l + 1] - rp[s * 32 + l]);
      off[s + 1] = off[s] + w * 32;
   }
   std::vector<int> sci((size_t)off[slices], 0);
   std::vector<double> sva((size_t)off[slices], 0.0), ssv((size_t)off[slices], 0.0);
   for (int r = 0; r < nrows; r++)
      for (int k = 0; k < rp[r + 1] - rp[r]; k++) {
         const size_t d = (size_t)off[r / 32] + (size_t)k * 32 + (r & 31);
         sci[d] = ci[rp[r] + k]; sva[d] = va[rp[r] + k]; ssv[d] = sv[rp[r] + k];
      }
   std::vector<std::vector<SuGrp>> gs;
   sellu_encode_chunk(nrows, off.data(), rp, 0, slices, 0, sci.data(), sva.data(), ssv.data(), gs);
   SuTable tab;
   int *desc = (int *)malloc(sizeof(int) * 2 * std::max<size_t>((size_t)slices, 1));
   for (int s = 0; s < slices; s++) {
      const int2 d = tab.add(gs[(size_t)s]);
      desc[2 * s] = d.x; desc[2 * s + 1] = d.y;
   }
   const size_t tot = tab.groups.size();
   int *dl = (int *)malloc(sizeof(int) * std::max<size_t>(tot, 1));
   unsigned int *mk = (unsigned int *)malloc(sizeof(unsigned int) * std::max<size_t>(tot, 1));
   double *gv = (double *)malloc(sizeof(double) * std::max<size_t>(tot, 1));
   double *gsvp = (double *)malloc(sizeof(double) * std::max<size_t>(tot, 1));
   for (size_t q = 0; q < tot; q++) { dl[q] = tab.groups[q].delta; mk[q] = tab.groups[q].mask; gv[q] = tab.groups[q].va; gsvp[q] = tab.groups[q].sv; }
   *desc_out = desc; *delta_out = dl; *mask_out = mk; *gva_out = gv; *gsv_out = gsvp; *ngroups = (int)tot;
   return slices;
}
void amgb_host_free(void *p) { free(p); }

// Row chunks of the warp-stream kernel: consecutive rows whose entries fit AMGB_WARP_CHUNK (and at most AMGB_WARP_CHUNK
// rows); a longer row is a chunk of its own.
static int build_stream_blocks(amgb_ctx *c, DevCSR &M, int nrows, const int *rp)
{
   std::vector<int4> blk;
   blk.reserve((size_t)rp[nrows] / 1024 + 16);
   int r = 0;
   while (r < nrows) {
      const int start = r;
      while (r < nrows && r - start < AMGB_WARP_CHUNK && rp[r + 1] - rp[start] <= AMGB_WARP_CHUNK) r++;
      if (r == start) r++;
      blk.push_back(make_int4(start, r, rp[start], rp[r]));
   }
   c->last_blk = blk;
   int4 *d_blk;
   int rc;
   if ((rc = dev_upload(c, &d_blk, blk.data(), blk.size()))) return rc;
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   M.nblk = (int)blk.size();
   M.blk = d_blk;
   return AMGB_OK;
}

int amgb_set_matrix(amgb_ctx *c, int kind, int level, int nrows, int ncols, int nnz,
                    const int *rp, const int *ci, const double *va)
{
   if (!c || !rp || (nnz > 0 && (!ci || !va))) return amgb_fail(c, AMGB_EINVAL, "null matrix arrays");
   // layout conversion below is OpenMP-parallel; launchers such as torchrun export OMP_NUM_THREADS=1
   if (omp_get_max_threads() < c->host_threads) omp_set_num_threads(c->host_threads);
   if (c->L == 0) return amgb_fail(c, AMGB_ESTATE, "call amgb_set_num_levels first");
   if (level < 0 || level >= c->L || (kind != AMGB_MAT_A && level >= c->L - 1 && c->L > 1))
      return amgb_fail(c, AMGB_EINVAL, "level %d out of range for kind %d", level, kind);
   if (nrows < 0 || ncols < 0 || nnz < 0 || rp[0] != 0 || rp[nrows] != nnz) return amgb_fail(c, AMGB_EINVAL, "inconsistent CSR");
   CUDA_OK(c, cudaSetDevice(c->device));
   DevCSR &M = kind == AMGB_MAT_A ? c->A[level] : (kind == AMGB_MAT_P ? c->P[level] : c->R[level]);
   if (M.rp) return amgb_fail(c, AMGB_ESTATE, "matrix (kind %d, level %d) already set", kind, level);
   if (kind == AMGB_MAT_A) {
      if (nrows != ncols && !c->dist) return amgb_fail(c, AMGB_EINVAL, "A must be square");
      const int doff = amgb_dist_diag_offset(c, level);   // local row block of a partitioned level: extended numbering
      for (int r = 0; r < nrows; r++)
         if (rp[r + 1] > rp[r] && ci[rp[r]] != r + doff) return amgb_fail(c, AMGB_EINVAL, "A_%d row %d is not diagonal-first", level, r);
   }
   int *d_rp, *d_ci; double *d_va;
   int rc;
   // coarse levels (level >= 2, everything of the matrix fits in what is left of the arena) live in the L2-pinned arena
   c->alloc_in_arena = c->opt.l2_persist && level >= 2 && (size_t)nnz * 40 + (size_t)nrows * 16 + 65536 <= c->arena_size - c->arena_used;
   struct ArenaOff { amgb_ctx *c; ~ArenaOff() { c->alloc_in_arena = false; } } arena_off{c};
   if ((rc = dev_upload(c, &d_rp, rp, (size_t)nrows + 1))) return rc;
   M.nrows = nrows; M.ncols = ncols; M.nnz = nnz;
   M.rp = d_rp;
   M.lpr = pick_lpr(nrows, nnz);
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   if (c->opt.use_sell && nrows >= 1024) {
      if ((rc = build_sell(c, M, nrows, rp, ci, va, 1, 0.15))) return rc;
      // small levels stay on the warp-stream kernel: with few slices the one-row-per-lane loop is latency bound
      if (M.sell_slices == 0 && c->opt.sell_sigma > 1 && nrows >= 262144 && (double)nnz / nrows < 96.0) {
         if ((rc = build_sell(c, M, nrows, rp, ci, va, c->opt.sell_sigma, 0.25))) return rc;
      }
   }
   // lean storage (amgb_options.lean_storage): a matrix that lives in sliced ELL keeps NO second copy in CSR -- only the row
   // pointer stays (the SELL-U encoder and the long-row test read it).  The CSR arrays are what the Gauss-Seidel-type
   // smoothers, the transposed product and the set-up kernels (diagonal, l1 norms) read, so lean storage is limited to
   // the (L1-)Jacobi family and the diagonal / l1 norms of an A_l are formed here, on the host, instead.
   const bool jac = c->opt.smoother == AMGB_SMOOTH_JACOBI || c->opt.smoother == AMGB_SMOOTH_L1_JACOBI;
   const bool lean = c->opt.lean_storage && jac && M.sell_slices > 0;
   d_ci = nullptr; d_va = nullptr;
   if (!lean) {
      if ((rc = dev_upload(c, &d_ci, ci, (size_t)nnz))) return rc;
      if ((rc = dev_upload(c, &d_va, va, (size_t)nnz))) return rc;
      CUDA_OK(c, cudaStreamSynchronize(c->stream));
   } else if (kind == AMGB_MAT_A) {
      std::vector<double> hd((size_t)nrows), hl((size_t)nrows);
#pragma omp parallel for schedule(static)
      for (int r = 0; r < nrows; r++) {
         double sabs = 0.0;
         for (int p = rp[r]; p < rp[r + 1]; p++) sabs += fabs(va[p]);
         hl[r] = sabs;
         hd[r] = rp[r + 1] > rp[r] ? va[rp[r]] : 0.0;
      }
      double *dd = nullptr, *dl = nullptr;
      if ((rc = dev_upload(c, &dd, hd.data(), hd.size()))) return rc;
      if ((rc = dev_upload(c, &dl, hl.data(), hl.size()))) return rc;
      CUDA_OK(c, cudaStreamSynchronize(c->stream));
      c->lean_diag[level] = dd;
      c->lean_l1[level] = dl;
   }
   M.ci = d_ci; M.va = d_va;
   // long rows (restrictions on coarse levels: 150-300 entries) are served best by one warp per row; everything
   // shorter goes through the stream kernel (measured per matrix with tools/spmv_sweep.py, profiles/)
   const bool long_rows = nrows > 0 && (double)nnz / nrows >= 96.0;
   if (long_rows) M.lpr = 32;
   if (c->opt.use_stream && M.sell_slices == 0 && nrows > 0 && !long_rows) {
      if ((rc = build_stream_blocks(c, M, nrows, rp))) return rc;
   }
   // DMEM convention: dense inverse of the coarsest operator (hypre_GaussElimSetup, src/DMEM_Setup.cpp:385-388),
   // applied later as one full SpMV
   if (kind == AMGB_MAT_A && level == c->L - 1 && c->opt.coarse_solve && c->L > 1) {
      const int n = nrows;
      if (n > 2048) return amgb_fail(c, AMGB_EINVAL, "coarsest level has %d rows: too large for the dense direct solve", n);
      std::vector<double> Mx((size_t)n * 2 * n, 0.0);         // [A | I]
      for (int i = 0; i < n; i++) {
         for (int p = rp[i]; p < rp[i + 1]; p++) Mx[(size_t)i * 2 * n + ci[p]] += va[p];
         Mx[(size_t)i * 2 * n + n + i] = 1.0;
      }
      for (int k = 0; k < n; k++) {                            // Gauss-Jordan, partial pivoting
         int piv = k;
         for (int i = k + 1; i < n; i++)
            if (fabs(Mx[(size_t)i * 2 * n + k]) > fabs(Mx[(size_t)piv * 2 * n + k])) piv = i;
         if (Mx[(size_t)piv * 2 * n + k] == 0.0) return amgb_fail(c, AMGB_EINVAL, "coarsest operator is singular");
         if (piv != k)
            for (int j = 0; j < 2 * n; j++) std::swap(Mx[(size_t)k * 2 * n + j], Mx[(size_t)piv * 2 * n + j]);
         const double d = 1.0 / Mx[(size_t)k * 2 * n + k];
         for (int j = 0; j < 2 * n; j++) Mx[(size_t)k * 2 * n + j] *= d;
         for (int i = 0; i < n; i++) {
            if (i == k) continue;
            const double fct = Mx[(size_t)i * 2 * n + k];
            if (fct != 0.0)
               for (int j = 0; j < 2 * n; j++) Mx[(size_t)i * 2 * n + j] -= fct * Mx[(size_t)k * 2 * n + j];
         }
      }
      std::vector<int> irp((size_t)n + 1), ici((size_t)n * n);
      std::vector<double> iva((size_t)n * n);
      for (int i = 0; i <= n; i++) irp[i] = i * n;
      for (int i = 0; i < n; i++)
         for (int j = 0; j < n; j++) { ici[(size_t)i * n + j] = j; iva[(size_t)i * n + j] = Mx[(size_t)i * 2 * n + n + j]; }
      int *d_irp, *d_ici; double *d_iva;
      if ((rc = dev_upload(c, &d_irp, irp.data(), irp.size()))) return rc;
      if ((rc = dev_upload(c, &d_ici, ici.data(), ici.size()))) return rc;
      if ((rc = dev_upload(c, &d_iva, iva.data(), iva.size()))) return rc;
      CUDA_OK(c, cudaStreamSynchronize(c->stream));
      c->Ainv = DevCSR();
      c->Ainv.nrows = n; c->Ainv.ncols = n; c->Ainv.nnz = n * n;
      c->Ainv.rp = d_irp; c->Ainv.ci = d_ici; c->Ainv.va = d_iva; c->Ainv.lpr = 32;
   }
   // multi-GPU: which launch units touch only owned entries of the input vector (see DevCSR::ulo/uhi)
   int c0 = 0, c1 = 0;
   if (amgb_dist_owned_cols(c, kind, level, &c0, &c1) && nrows > 0) {
      std::vector<char> rint((size_t)nrows, 1);
#pragma omp parallel for schedule(static)
      for (int r = 0; r < nrows; r++)
         for (int p = rp[r]; p < rp[r + 1]; p++)
            if (ci[p] < c0 || ci[p] >= c1) { rint[r] = 0; break; }
      const int nu = spmv_units(M);
      std::vector<char> uint_((size_t)nu, 1);
      if (M.sell_slices > 0) {
         for (int u = 0; u < nu; u++)
            for (int l = 0; l < 32; l++) {
               const int slot = u * 32 + l;
               const int r = M.sell_perm ? c->last_perm[slot] : (slot < nrows ? slot : -1);
               if (r >= 0 && !rint[r]) { uint_[u] = 0; break; }
            }
      } else if (M.nblk > 0) {
         for (int u = 0; u < nu; u++)
            for (int r = c->last_blk[u].x; r < c->last_blk[u].y; r++)
               if (!rint[r]) { uint_[u] = 0; break; }
      } else {
         for (int u = 0; u < nu; u++) uint_[u] = rint[u];
      }
      // the longest run of interior units (near the slab faces interior and boundary units interleave; the units
      // outside the run simply wait for the exchange)
      int lo = 0, hi = 0;
      for (int u = 0; u < nu;) {
         if (!uint_[u]) { u++; continue; }
         int v = u;
         while (v < nu && uint_[v]) v++;
         if (v - u > hi - lo) { lo = u; hi = v; }
         u = v;
      }
      const bool contiguous = hi > lo;
      if (contiguous) { M.ulo = lo; M.uhi = hi; }
      if (getenv("AMGB_DEBUG"))
         fprintf(stderr, "[amgb] kind %d level %d: %d units (%s), owned cols [%d,%d), interior units [%d,%d) contiguous=%d\n", kind, level, nu,
                 M.sell_slices > 0 ? (M.sell_perm ? "sell-sigma" : "sell") : (M.nblk > 0 ? "chunks" : "rows"), c0, c1, lo, hi, (int)contiguous);
   } else if (getenv("AMGB_DEBUG") && c->dist) {
      fprintf(stderr, "[amgb] kind %d level %d: input vector not partitioned, no split\n", kind, level);
   }
   return AMGB_OK;
}

// ---- setup ----------------------------------------------------------------------------------------
int amgb_setup(amgb_ctx *c)
{
   if (!c) return AMGB_EINVAL;
   if (c->ready) return amgb_fail(c, AMGB_ESTATE, "setup already done");
   const int L = c->L;
   if (L == 0) return amgb_fail(c, AMGB_ESTATE, "no hierarchy");
   for (int l = 0; l < L; l++) {
      if (!c->A[l].rp) return amgb_fail(c, AMGB_ESTATE, "A_%d missing", l);
      if (l < L - 1) {
         if (!c->P[l].rp || !c->R[l].rp) return amgb_fail(c, AMGB_ESTATE, "P_%d / R_%d missing", l, l);
         if (!c->dist && (c->P[l].nrows != c->A[l].nrows || c->P[l].ncols != c->A[l + 1].nrows ||
                          c->R[l].nrows != c->A[l + 1].nrows || c->R[l].ncols != c->A[l].nrows))
            return amgb_fail(c, AMGB_EINVAL, "transfer shapes at level %d do not match", l);
      }
   }
   CUDA_OK(c, cudaSetDevice(c->device));
   const amgb_options &o = c->opt;
   const bool multadd = o.solver == AMGB_SOLVER_MULTADD || o.solver == AMGB_SOLVER_ASYNC_MULTADD;
   c->symmetric = multadd && o.num_pre_smooth_sweeps > 0 && o.num_post_smooth_sweeps > 0 &&
                  (o.smoother == AMGB_SMOOTH_JACOBI || o.smoother == AMGB_SMOOTH_L1_JACOBI);
   if (o.smoother == AMGB_SMOOTH_L1_HYBRID_JGS && o.solver != AMGB_SOLVER_BPX)
      return amgb_fail(c, AMGB_EINVAL, "L1_HYBRID_JACOBI_GAUSS_SEIDEL exists in the Parfor smoother only (BPX); the reference's ALL_LEVELS "
                                       "dispatcher silently runs weighted Jacobi for it (src/SMEM_Solve.cpp:277-323)");
   if (o.factor_restriction && !(o.solver == AMGB_SOLVER_MULTADD && c->symmetric && o.factor_level0 && o.num_fine_smooth_sweeps == 1 && !c->dist))
      return amgb_fail(c, AMGB_EINVAL, "factor_restriction applies to synchronous Multadd on one GPU with factor_level0, the symmetrised "
                                       "(L1-)Jacobi smoother and num_fine_smooth_sweeps = 1");
   if (o.factor_level0 && !((o.solver == AMGB_SOLVER_MULTADD || o.solver == AMGB_SOLVER_ASYNC_MULTADD) && c->symmetric))
      return amgb_fail(c, AMGB_EINVAL, "factor_level0 applies to Multadd with the symmetrised (L1-)Jacobi smoother");
   int rc;
   c->ws.assign(L, nullptr); c->dow.assign(L, nullptr); c->l1.assign(L, nullptr); c->inv_l1.assign(L, nullptr);
   c->r.assign(L, nullptr); c->e.assign(L, nullptr); c->t.assign(L, nullptr); c->w.assign(L, nullptr);
   int maxn = 0;
   for (int l = 0; l < L; l++) {
      const int n = c->A[l].nrows;
      maxn = std::max(maxn, n);
      if ((rc = dev_alloc(c, &c->ws[l], n))) return rc;
      if ((rc = dev_alloc(c, &c->dow[l], n))) return rc;
      if ((rc = dev_alloc(c, &c->l1[l], n))) return rc;
      if ((rc = dev_alloc(c, &c->inv_l1[l], n))) return rc;
      const bool lean = c->A[l].va == nullptr && c->A[l].nnz > 0;     // lean storage: sliced ELL only, diagonal / l1 came from the host
      if (lean) {
         c->launches += launch_diag_scale_vec(c->stream, n, c->lean_diag[l], c->lean_l1[l], o.smooth_weight, c->ws[l], c->dow[l], c->l1[l], c->inv_l1[l]);
      } else {
         c->launches += launch_diag_scale(c->stream, c->A[l], o.smooth_weight, c->ws[l], c->dow[l]);
         c->launches += launch_l1(c->stream, c->A[l], c->l1[l], c->inv_l1[l]);
      }
      // column-scaled copy of A's values for the one-pass symmetrised smoother
      double *sv = nullptr;
      const double *cs = (o.smoother == AMGB_SMOOTH_L1_JACOBI) ? c->inv_l1[l] : c->ws[l];
      // (a partitioned level's columns are in the rank's extended numbering: amgb_dist_setup fills sval there)
      const bool part = amgb_dist_level_distributed(c, l);
      if (!lean) {
         if ((rc = dev_alloc(c, &sv, (size_t)c->A[l].nnz))) return rc;
         if (!part) c->launches += launch_colscale(c->stream, c->A[l].nnz, c->A[l].ci, c->A[l].va, cs, sv);
      }
      c->A[l].sval = sv;
      if (c->A[l].sell_slices > 0) {
         long pe = c->sell_entries[&c->A[l]];
         double *ssv = nullptr;
         if ((rc = dev_alloc(c, &ssv, (size_t)pe))) return rc;
         if (!part) c->launches += launch_colscale(c->stream, (int)pe, c->A[l].sell_ci, c->A[l].sell_va, cs, ssv);
         c->A[l].sell_sval = ssv;
      }
      if (!part && (rc = build_sellu(c, c->A[l]))) return rc;
      if ((rc = dev_zero(c, &c->r[l], n))) return rc;
      if ((rc = dev_zero(c, &c->e[l], n))) return rc;
      if ((rc = dev_zero(c, &c->t[l], n))) return rc;
      if ((rc = dev_zero(c, &c->w[l], n))) return rc;
   }
   const int n0 = c->A[0].nrows;
   if ((rc = dev_zero(c, &c->f, n0))) return rc;
   if ((rc = dev_zero(c, &c->u, n0))) return rc;
   if ((rc = dev_zero(c, &c->cvec, n0))) return rc;
   if ((rc = dev_zero(c, &c->u_outer, n0))) return rc;
   if ((rc = dev_zero(c, &c->y_outer, n0))) return rc;
   for (int l = 0; l < L; l++) {            // (a partitioned level's matrices have more columns than rows: ghosts)
      maxn = std::max(maxn, c->A[l].ncols);
      if (l < L - 1) maxn = std::max(maxn, std::max(std::max(c->P[l].ncols, c->P[l].nrows), std::max(c->R[l].ncols, c->R[l].nrows)));
   }
   c->io_len = maxn;
   if ((rc = dev_zero(c, &c->io_a, maxn))) return rc;
   if ((rc = dev_zero(c, &c->io_b, maxn))) return rc;
   if ((rc = dev_zero(c, &c->io_c, maxn))) return rc;
   c->npartials = c->cfg.num_sms * c->cfg.ctas_per_sm;
   if ((rc = dev_zero(c, &c->partials, c->npartials))) return rc;
   if ((rc = dev_zero(c, &c->d_scalars, 64))) return rc;
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   c->ready = true;
   return AMGB_OK;
}

// ---- vectors --------------------------------------------------------------------------------------
int amgb_set_rhs(amgb_ctx *c, const double *f)
{
   NEED_READY(c);
   if (!f) return amgb_fail(c, AMGB_EINVAL, "null rhs");
   CUDA_OK(c, cudaMemcpyAsync(c->f, f, sizeof(double) * c->A[0].nrows, cudaMemcpyHostToDevice, c->stream));
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   return AMGB_OK;
}
int amgb_set_solution(amgb_ctx *c, const double *u)
{
   NEED_READY(c);
   if (u) CUDA_OK(c, cudaMemcpyAsync(c->u, u, sizeof(double) * c->A[0].nrows, cudaMemcpyHostToDevice, c->stream));
   else CUDA_OK(c, cudaMemsetAsync(c->u, 0, sizeof(double) * c->A[0].nrows, c->stream));
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   return AMGB_OK;
}
int amgb_get_solution(amgb_ctx *c, double *u)
{
   NEED_READY(c);
   CUDA_OK(c, cudaMemcpyAsync(u, c->u, sizeof(double) * c->A[0].nrows, cudaMemcpyDeviceToHost, c->stream));
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   return AMGB_OK;
}
int amgb_get_residual(amgb_ctx *c, double *r)
{
   NEED_READY(c);
   CUDA_OK(c, cudaMemcpyAsync(r, c->r[0], sizeof(double) * c->A[0].nrows, cudaMemcpyDeviceToHost, c->stream));
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   return AMGB_OK;
}

}  // extern "C"

int amgb_build_sellu(amgb_ctx *c, DevCSR &M) { return build_sellu(c, M); }

// ---- enqueue helpers (no host synchronisation) ---------------------------------------------------
static inline SpmvEpilogue epi(double alpha, double beta, const double *b, double gamma = 0.0, const double *cc = nullptr,
                               const double *rs = nullptr)
{
   SpmvEpilogue e;
   e.alpha = alpha; e.beta = beta; e.gamma = gamma; e.b = b; e.c = cc; e.rs = rs;
   return e;
}

void enq_spmv(amgb_ctx *c, const DevCSR &M, bool sval, const double *x, double *y, const SpmvEpilogue &e, bool norm)
{
   int grid = 0;
   c->launches += launch_spmv(c->cfg, c->stream, M, sval, x, y, e, norm ? c->partials : nullptr, &grid);
   if (norm) c->launches += launch_reduce_partials(c->stream, c->partials, grid, c->d_scalars);
}

// the same with the fused sum_i y_i w_i reduced into *dot_out (w == nullptr: plain enq_spmv, no reduction)
void enq_spmv_dot(amgb_ctx *c, const DevCSR &M, bool sval, const double *x, double *y, const SpmvEpilogue &e, const double *w, double *dot_out)
{
   if (!w) { enq_spmv(c, M, sval, x, y, e, false); return; }
   int grid = 0;
   c->launches += launch_spmv(c->cfg, c->stream, M, sval, x, y, e, c->partials, &grid, w);
   c->launches += launch_reduce_partials(c->stream, c->partials, grid, dot_out);
}

// *out = sum_i x_i w_i (nothing when w == nullptr)
static void enq_dot(amgb_ctx *c, int n, const double *x, const double *w, double *out)
{
   if (!w) return;
   int grid = 0;
   c->launches += launch_dot(c->cfg, c->stream, n, x, w, c->partials, &grid);
   c->launches += launch_reduce_partials(c->stream, c->partials, grid, out);
}

// r0 = f - A0 u, d_scalars[0] = ||r||^2     (SMEM_Sync_Residual + norm, src/SMEM_Solve.cpp:192-203)
void enq_residual(amgb_ctx *c)
{
   enq_spmv(c, c->A[0], false, c->u, c->r[0], epi(-1.0, 1.0, c->f), true);
}


// one hybrid Jacobi / Gauss-Seidel sweep on level l: the explicit block list when one was given (amgb_set_jgs_blocks), else the
// uniform blocks of opt.jgs_block_rows
static int jgs_sweep(amgb_ctx *c, int l, const DevCSR &A, const double *f, double *u, const double *u_prev, const double *scale, bool zero)
{
   if (l >= 0 && l < (int)c->jgs_bounds.size() && c->jgs_bounds[l])
      return launch_hybrid_jgs_list(c->cfg, c->stream, A, f, u, u_prev, scale, c->jgs_bounds[l], c->jgs_nb[l], zero);
   return launch_hybrid_jgs(c->cfg, c->stream, A, f, u, u_prev, scale, c->opt.jgs_block_rows, zero);
}

// e = S_l f from a zero initial guess, `sweeps` sweeps; scratch: t[l], w[l] are free to use.
// Dispatch as SMEM_Smooth (src/SMEM_Solve.cpp:264-377).  parfor: the ONE_LEVEL branch (BPX).
void enq_smooth_zero(amgb_ctx *c, int l, const double *f, double *e, int sweeps, bool symmetric, bool parfor,
                     double *s1, double *s2)
{
   const DevCSR &A = c->A[l];
   const int n = A.nrows;
   const int sm = c->opt.smoother;
   if (sweeps < 1) { cudaMemsetAsync(e, 0, sizeof(double) * n, c->stream); return; }
   if (sm == AMGB_SMOOTH_ASYNC_GS || sm == AMGB_SMOOTH_SEMI_ASYNC_GS) {
      // chaotic Gauss-Seidel from the zero guess the additive cycles give it (src/SMEM_Smooth.cpp:445-502)
      cudaMemsetAsync(e, 0, sizeof(double) * n, c->stream);
      c->launches += launch_async_gs(c->cfg, c->stream, A, f, e, c->opt.jgs_block_rows, sweeps, sm == AMGB_SMOOTH_SEMI_ASYNC_GS);
      return;
   }
   if (sm == AMGB_SMOOTH_HYBRID_JGS || sm == AMGB_SMOOTH_L1_HYBRID_JGS) {
      // Parfor branch (BPX): divisor A_diag = a_ii / w, or the l1 norms for L1_HYBRID_JACOBI_GAUSS_SEIDEL (src/SMEM_Smooth.cpp:253-263)
      const double *scale = sm == AMGB_SMOOTH_L1_HYBRID_JGS ? c->l1[l] : (parfor ? c->dow[l] : nullptr);
      c->launches += jgs_sweep(c, l, A, f, e, nullptr, scale, true);
      for (int k = 1; k < sweeps; k++) {
         cudaMemcpyAsync(s1, e, sizeof(double) * n, cudaMemcpyDeviceToDevice, c->stream);
         c->launches += jgs_sweep(c, l, A, f, e, s1, scale, false);
      }
      return;
   }
   const double *rs = (sm == AMGB_SMOOTH_L1_JACOBI) ? c->inv_l1[l] : c->ws[l];
   if (symmetric) {
      // sweep 1: e = rs.*(2f - (A*diag(rs)) f)      (src/SMEM_Smooth.cpp:655-695 in one pass)
      enq_spmv(c, A, true, f, e, epi(-1.0, 2.0, f, 0.0, nullptr, rs), false);
      for (int k = 1; k < sweeps; k++) {
         // reference: r = f - A u; then the same update with zero_flags still 1 -> u = S r (:685-701)
         enq_spmv(c, A, false, e, s1, epi(-1.0, 1.0, f), false);
         enq_spmv(c, A, true, s1, e, epi(-1.0, 2.0, s1, 0.0, nullptr, rs), false);
      }
      return;
   }
   // (L1-)Jacobi: sweep 1 from zero guess u = rs.*f (src/SMEM_Smooth.cpp:381-389,422-426); then
   // u <- u + rs.*(f - A u_prev) with ping-pong buffers, arranged so that the result lands in e
   double *cur = ((sweeps - 1) & 1) ? s1 : e;
   double *oth = (cur == e) ? s1 : e;
   c->launches += launch_scale(c->cfg, c->stream, n, rs, f, cur);
   for (int k = 1; k < sweeps; k++) {
      enq_spmv(c, A, false, cur, oth, epi(-1.0, 1.0, f, 1.0, cur, rs), false);
      std::swap(cur, oth);
   }
   (void)s2;
}

// One additive cycle on residual r[0]:  target = gamma*target + B r.  r[0] is read and never written (the factorised level-0
// path included): the preconditioned conjugate-gradient solve (pcg.cu) keeps its residual there across the cycle.
// dot_w != nullptr: sum_i target_i dot_w_i is reduced into *dot_out, fused into the cycle's last launch when that is an SpMV.
void enq_cycle(amgb_ctx *c, double *target, bool accumulate, const double *dot_w, double *dot_out)
{
   const int L = c->L;
   const amgb_options &o = c->opt;
   const int n0 = c->A[0].nrows;
   const int solver = o.solver;
   const bool multadd = solver == AMGB_SOLVER_MULTADD || solver == AMGB_SOLVER_ASYNC_MULTADD;
   const bool afacx = solver == AMGB_SOLVER_AFACX || solver == AMGB_SOLVER_ASYNC_AFACX;
   const bool bpx = solver == AMGB_SOLVER_BPX;
   if (L == 1) {
      // single level: Multadd/AFACx coarsest contributes nothing; BPX smooths it
      if (bpx) {
         enq_smooth_zero(c, 0, c->r[0], c->e[0], o.num_pre_smooth_sweeps, false, true, c->t[0], c->w[0]);
         if (accumulate) c->launches += launch_add(c->cfg, c->stream, n0, c->e[0], target);
         else cudaMemcpyAsync(target, c->e[0], sizeof(double) * n0, cudaMemcpyDeviceToDevice, c->stream);
      } else if (!accumulate) cudaMemsetAsync(target, 0, sizeof(double) * n0, c->stream);
      enq_dot(c, n0, target, dot_w, dot_out);
      return;
   }
   // restriction chain, shared by all levels (the reference repeats it per level group,
   // src/SMEM_Sync_AMG.cpp:475-490; the result is identical)
   const bool direct = o.coarse_solve && c->Ainv.rp != nullptr;   // DMEM convention: e_{L-1} = A_{L-1}^{-1} r_{L-1}
   const int last_r = (multadd && !direct) ? L - 2 : L - 1;   // SMEM Multadd never reads r_{L-1} (coarsest contributes 0)
   // level-0 transfers in factorised form (amgb_options.factor_level0): t_0 = r_0 - A_0 diag(w/d) r_0 serves both
   // Rbar_0 r_0 = R_0 t_0 and the symmetrised smoother e_0 = (w/d) o (r_0 + t_0); on the way up
   // u += e_0 + Pbar_0 e_1 = (w/d) o (r_0 + t_0 - A_0 v) + v with v = P_0 e_1.  Two passes over A_0 (sliced ELL, HBM
   // speed) and two over the plain P_0 / R_0 replace A_0 + Pbar_0 + Rbar_0 (3.5x the entries of P_0, L1-bound).
   const bool fact0 = o.factor_level0 && multadd && c->symmetric && last_r >= 1;
   // the same on the levels 1 <= l < last_r (amgb_options.factor_restriction, one smoothing sweep): the smoother's pass over
   // A_l also writes t_l = r_l - A_l diag(s) r_l, and e_l = s o (r_l + t_l) comes out of it as a second output; then
   // Rbar_l r_l = R_l t_l with the plain R_l = P_l^T (about a fifth of Rbar_l's entries).  Same launches as the explicit form.
   const bool factr = fact0 && o.factor_restriction;
   for (int l = 0; l < last_r; l++) {
      if (fact0 && l == 0) {
         enq_spmv(c, c->A[0], true, c->r[0], c->t[0], epi(-1.0, 1.0, c->r[0]), false);        // t_0
         enq_spmv(c, c->R[0], false, c->t[0], c->r[1], epi(1.0, 0.0, nullptr), false);       // r_1 = R_0 t_0
      } else if (factr) {
         const double *rs = (o.smoother == AMGB_SMOOTH_L1_JACOBI) ? c->inv_l1[l] : c->ws[l];
         c->launches += launch_spmv(c->cfg, c->stream, c->A[l], true, c->r[l], c->t[l], epi(-1.0, 1.0, c->r[l]), nullptr, nullptr,
                                    nullptr, c->e[l], rs);                                     // t_l and e_l
         enq_spmv(c, c->R[l], false, c->t[l], c->r[l + 1], epi(1.0, 0.0, nullptr), false);   // r_{l+1} = R_l t_l
      } else enq_spmv(c, c->R[l], false, c->r[l], c->r[l + 1], epi(1.0, 0.0, nullptr), false);
   }
   // per-level corrections e_l (levels are independent)
   const int top = (bpx || direct) ? L : L - 1;  // BPX also smooths the coarsest level (:217-236)
   for (int l = 0; l < top; l++) {
      if (fact0 && l == 0) continue;                  // e_0 is folded into the last launch of the cycle
      if (factr && l < last_r) continue;              // e_l came with t_l
      if (direct && l == L - 1) enq_spmv(c, c->Ainv, false, c->r[l], c->e[l], epi(1.0, 0.0, nullptr), false);
      else if (multadd) enq_smooth_zero(c, l, c->r[l], c->e[l], o.num_fine_smooth_sweeps, c->symmetric, false, c->t[l], c->w[l]);
      else if (bpx) enq_smooth_zero(c, l, c->r[l], c->e[l], o.num_pre_smooth_sweeps, false, true, c->t[l], c->w[l]);
      else if (afacx) {
         // src/SEQ_AMG.cpp:172-208: u_c = S_{l+1} r_{l+1}; e = P u_c; r_f = r_l - A_l e; u_f = S_l r_f
         const int cl = l + 1;
         double *uc = c->t[cl];
         enq_smooth_zero(c, cl, c->r[cl], uc, o.num_coarse_smooth_sweeps, false, false, c->w[cl], c->e[cl]);
         enq_spmv(c, c->P[l], false, uc, c->t[l], epi(1.0, 0.0, nullptr), false);
         enq_spmv(c, c->A[l], false, c->t[l], c->w[l], epi(-1.0, 1.0, c->r[l]), false);
         // scratch for the fine smooth must not alias its input w[l] nor the pending e[l+1]
         enq_smooth_zero(c, l, c->w[l], c->e[l], o.num_fine_smooth_sweeps, false, false, c->t[l], c->t[l]);
      }
   }
   // Horner prolongation: c = e_0 + P_0 (e_1 + P_1 (e_2 + ...)), same sum as the reference's
   // per-level prolongation chains (src/SEQ_AMG.cpp:213-233)
   for (int l = top - 2; l >= 1; l--) enq_spmv(c, c->P[l], false, c->e[l + 1], c->e[l], epi(1.0, 1.0, c->e[l]), false);
   if (fact0) {
      // v = P_0 e_1;  target = [target +] v + (w/d) o (r_0 + t_0 - A_0 v)
      enq_spmv(c, c->P[0], false, c->e[1], c->w[0], epi(1.0, 0.0, nullptr), false);
      const double *rs0 = (o.smoother == AMGB_SMOOTH_L1_JACOBI) ? c->inv_l1[0] : c->ws[0];
      SpmvEpilogue fe = epi(-1.0, 1.0, c->r[0], 1.0, accumulate ? target : nullptr, rs0);
      fe.b2 = c->t[0]; fe.beta2 = 1.0;
      fe.xs = c->w[0]; fe.xself = 1.0;
      enq_spmv_dot(c, c->A[0], false, c->w[0], target, fe, dot_w, dot_out);
   } else if (top >= 2) {
      // target = [target +] e_0 + P_0 e_1   (u += e fused into the last prolongation)
      enq_spmv_dot(c, c->P[0], false, c->e[1], target, epi(1.0, 1.0, c->e[0], 1.0, accumulate ? target : nullptr), dot_w, dot_out);
   } else {
      if (accumulate) c->launches += launch_add(c->cfg, c->stream, n0, c->e[0], target);
      else cudaMemcpyAsync(target, c->e[0], sizeof(double) * n0, cudaMemcpyDeviceToDevice, c->stream);
      enq_dot(c, n0, target, dot_w, dot_out);
   }
}

// `sweeps` general (L1-)Jacobi sweeps u <- u + rs o (f - A u) in place (ping-pong through `scratch`)
static void enq_jacobi_sweeps(amgb_ctx *c, int l, const double *f, double *u, int sweeps, double *scratch)
{
   const DevCSR &A = c->A[l];
   const double *rs = (c->opt.smoother == AMGB_SMOOTH_L1_JACOBI) ? c->inv_l1[l] : c->ws[l];
   double *cur = u, *oth = scratch;
   for (int k = 0; k < sweeps; k++) {
      enq_spmv(c, A, false, cur, oth, epi(-1.0, 1.0, f, 1.0, cur, rs), false);
      std::swap(cur, oth);
   }
   if (cur != u) cudaMemcpyAsync(u, cur, sizeof(double) * A.nrows, cudaMemcpyDeviceToDevice, c->stream);
}

// One multiplicative V-cycle on (f, u) of level 0 -- SMEM_Sync_Parfor_Vcycle, src/SMEM_Sync_AMG.cpp:8-145 (the
// reference's comparator for the additive cycles; SURVEY.md 8f-2).  Level right-hand sides live in r[l], level
// solutions in e[l] (l >= 1).  As in the reference the first sweep on levels 1..L-2 starts from zero
// (zero_flags = 1 on the way down), and the coarsest level's num_pre + num_post sweeps continue from the
// value the previous cycle left there (its zero flag is never raised; e[L-1] is cleared at the start of a solve).
void enq_vcycle(amgb_ctx *c)
{
   const int L = c->L;
   const amgb_options &o = c->opt;
   for (int l = 0; l < L - 1; l++) {
      const double *fl = l == 0 ? c->f : c->r[l];
      double *ul = l == 0 ? c->u : c->e[l];
      if (l == 0) enq_jacobi_sweeps(c, 0, fl, ul, o.num_pre_smooth_sweeps, c->t[0]);
      else enq_smooth_zero(c, l, fl, ul, o.num_pre_smooth_sweeps, false, true, c->t[l], c->w[l]);
      enq_spmv(c, c->A[l], false, ul, c->w[l], epi(-1.0, 1.0, fl), false);                 // r_fine = f - A u
      enq_spmv(c, c->R[l], false, c->w[l], c->r[l + 1], epi(1.0, 0.0, nullptr), false);    // f_{l+1} = R r_fine
   }
   {
      const int cl = L - 1;
      // DMEM's comparator (DMEM_MultCycle, src/DMEM_Mult.cpp:207): direct solve on the coarsest level
      if (o.coarse_solve && cl > 0 && c->Ainv.rp != nullptr)
         enq_spmv(c, c->Ainv, false, c->r[cl], c->e[cl], epi(1.0, 0.0, nullptr), false);
      else
         enq_jacobi_sweeps(c, cl, cl == 0 ? c->f : c->r[cl], cl == 0 ? c->u : c->e[cl],
                           o.num_pre_smooth_sweeps + o.num_post_smooth_sweeps, c->t[cl]);
   }
   for (int l = L - 2; l >= 0; l--) {
      const double *fl = l == 0 ? c->f : c->r[l];
      double *ul = l == 0 ? c->u : c->e[l];
      enq_spmv(c, c->P[l], false, c->e[l + 1], ul, epi(1.0, 1.0, ul), false);              // u += P u_c
      enq_jacobi_sweeps(c, l, fl, ul, o.num_post_smooth_sweeps, c->t[l]);
   }
}

int amgb_fetch_scalar(amgb_ctx *c, double *out)
{
   CUDA_OK(c, cudaMemcpyAsync(c->h_scalars, c->d_scalars, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   *out = c->h_scalars[0];
   return AMGB_OK;
}

extern "C" {

// Explicit Gauss-Seidel blocks of the hybrid smoother on one level: bounds[0] = 0 <= ... <= bounds[nblocks] = n_level (an empty block = a thread left without rows).  The
// reference's block is a thread's row range (src/SMEM_Smooth.cpp:567-581 with the nnz-balanced split of src/SMEM_Setup.cpp:954-959),
// so its results depend on the thread count; with this list the device sweeps the very same blocks.  nblocks = 0 returns to the
// uniform blocks of opt.jgs_block_rows.  Synchronous cycles and amgb_smooth only.
int amgb_set_jgs_blocks(amgb_ctx *c, int level, int nblocks, const int *bounds)
{
   if (!c || level < 0 || level >= c->L) return amgb_fail(c, AMGB_EINVAL, "bad level");
   if (nblocks == 0) { c->jgs_bounds[level] = nullptr; c->jgs_nb[level] = 0; return AMGB_OK; }
   const int n = c->A[level].nrows;
   if (nblocks < 0 || !bounds || n <= 0) return amgb_fail(c, AMGB_EINVAL, "block list given before the level's matrix, or empty");
   if (bounds[0] != 0 || bounds[nblocks] != n) return amgb_fail(c, AMGB_EINVAL, "block list must run from 0 to the level's row count %d", n);
   for (int b = 0; b < nblocks; b++)
      if (bounds[b + 1] < bounds[b]) return amgb_fail(c, AMGB_EINVAL, "block list is decreasing at block %d", b);   // an EMPTY block is a thread without rows (small levels)
   int *dev = nullptr;
   int rc = amgb_dev_alloc_bytes(c, (void **)&dev, sizeof(int) * ((size_t)nblocks + 1), false);
   if (rc) return rc;
   CUDA_OK(c, cudaMemcpyAsync(dev, bounds, sizeof(int) * ((size_t)nblocks + 1), cudaMemcpyHostToDevice, c->stream));
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   c->jgs_bounds[level] = dev;
   c->jgs_nb[level] = nblocks;
   if (c->graph_exec) { cudaGraphExecDestroy(c->graph_exec); c->graph_exec = nullptr; }     // the captured cycle held the old launches
   if (c->pcg_graph) { cudaGraphExecDestroy(c->pcg_graph); c->pcg_graph = nullptr; }
   return AMGB_OK;
}

// ---- per-op entry points (host in / host out) ------------------------------------------------------
int amgb_spgemv(amgb_ctx *c, int kind, int level, double alpha, const double *x, double beta, const double *b, double *y)
{
   NEED_READY(c);
   if (level < 0 || level >= c->L || (kind != AMGB_MAT_A && level >= c->L - 1)) return amgb_fail(c, AMGB_EINVAL, "bad level");
   const DevCSR &M = kind == AMGB_MAT_A ? c->A[level] : (kind == AMGB_MAT_P ? c->P[level] : c->R[level]);
   if (!x || !y || (beta != 0.0 && !b)) return amgb_fail(c, AMGB_EINVAL, "null vector");
   if (M.nrows > c->io_len || M.ncols > c->io_len) return amgb_fail(c, AMGB_EINVAL, "matrix larger than the staging vectors");
   CUDA_OK(c, cudaMemcpyAsync(c->io_a, x, sizeof(double) * M.ncols, cudaMemcpyHostToDevice, c->stream));
   if (beta != 0.0) CUDA_OK(c, cudaMemcpyAsync(c->io_b, b, sizeof(double) * M.nrows, cudaMemcpyHostToDevice, c->stream));
   enq_spmv(c, M, false, c->io_a, c->io_c, epi(alpha, beta, beta != 0.0 ? c->io_b : nullptr), false);
   CUDA_OK(c, cudaMemcpyAsync(y, c->io_c, sizeof(double) * M.nrows, cudaMemcpyDeviceToHost, c->stream));
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   CUDA_OK(c, cudaGetLastError());
   return AMGB_OK;
}

int amgb_spgemv_transpose(amgb_ctx *c, int kind, int level, const double *x, double *y)
{
   NEED_READY(c);
   if (level < 0 || level >= c->L || (kind != AMGB_MAT_A && level >= c->L - 1)) return amgb_fail(c, AMGB_EINVAL, "bad level");
   const DevCSR &M = kind == AMGB_MAT_A ? c->A[level] : (kind == AMGB_MAT_P ? c->P[level] : c->R[level]);
   if (!x || !y) return amgb_fail(c, AMGB_EINVAL, "null vector");
   if (M.nrows > c->io_len || M.ncols > c->io_len) return amgb_fail(c, AMGB_EINVAL, "matrix larger than the staging vectors");
   if (!M.ci && M.nnz > 0) return amgb_fail(c, AMGB_EINVAL, "the transposed product reads the CSR arrays, which lean storage does not keep");
   CUDA_OK(c, cudaMemcpyAsync(c->io_a, x, sizeof(double) * M.nrows, cudaMemcpyHostToDevice, c->stream));
   c->launches += launch_spmv_transpose(c->cfg, c->stream, M, c->io_a, c->io_c);
   CUDA_OK(c, cudaMemcpyAsync(y, c->io_c, sizeof(double) * M.ncols, cudaMemcpyDeviceToHost, c->stream));
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   CUDA_OK(c, cudaGetLastError());
   return AMGB_OK;
}

int amgb_smooth(amgb_ctx *c, int level, int smoother, int symmetric, int sweeps, int zero_guess, const double *f, double *u)
{
   NEED_READY(c);
   if (level < 0 || level >= c->L || !f || !u || sweeps < 1) return amgb_fail(c, AMGB_EINVAL, "bad smooth arguments");
   if (smoother != c->opt.smoother) return amgb_fail(c, AMGB_EINVAL, "smoother %d differs from the one set up (%d)", smoother, c->opt.smoother);
   const DevCSR &A = c->A[level];
   const int n = A.nrows;
   CUDA_OK(c, cudaMemcpyAsync(c->io_a, f, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
   if (zero_guess) {
      enq_smooth_zero(c, level, c->io_a, c->io_b, sweeps, symmetric != 0, false, c->io_c, c->w[level]);
   } else {
      // general sweeps from a given u (src/SMEM_Smooth.cpp:391-402,428-439,565-581)
      CUDA_OK(c, cudaMemcpyAsync(c->io_b, u, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
      if (symmetric) return amgb_fail(c, AMGB_EINVAL, "symmetrised smoother is only used from a zero guess");
      double *cur = c->io_b, *oth = c->io_c;
      for (int k = 0; k < sweeps; k++) {
         if (smoother == AMGB_SMOOTH_ASYNC_GS || smoother == AMGB_SMOOTH_SEMI_ASYNC_GS) {
            c->launches += launch_async_gs(c->cfg, c->stream, A, c->io_a, cur, c->opt.jgs_block_rows, 1, true);
         } else if (smoother == AMGB_SMOOTH_HYBRID_JGS) {
            CUDA_OK(c, cudaMemcpyAsync(oth, cur, sizeof(double) * n, cudaMemcpyDeviceToDevice, c->stream));
            c->launches += jgs_sweep(c, level, A, c->io_a, cur, oth, nullptr, false);
         } else {
            const double *rs = (smoother == AMGB_SMOOTH_L1_JACOBI) ? c->inv_l1[level] : c->ws[level];
            enq_spmv(c, A, false, cur, oth, epi(-1.0, 1.0, c->io_a, 1.0, cur, rs), false);
            std::swap(cur, oth);
         }
      }
      if (cur != c->io_b) CUDA_OK(c, cudaMemcpyAsync(c->io_b, cur, sizeof(double) * n, cudaMemcpyDeviceToDevice, c->stream));
   }
   CUDA_OK(c, cudaMemcpyAsync(u, c->io_b, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   CUDA_OK(c, cudaGetLastError());
   return AMGB_OK;
}

int amgb_norm2(amgb_ctx *c, const double *x, int n, double *out)
{
   NEED_READY(c);
   int maxn = 0;
   for (auto &a : c->A) maxn = std::max(maxn, a.nrows);
   if (!x || !out || n < 0 || n > maxn) return amgb_fail(c, AMGB_EINVAL, "bad norm2 arguments");
   CUDA_OK(c, cudaMemcpyAsync(c->io_a, x, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
   int grid = 0;
   c->launches += launch_sumsq(c->cfg, c->stream, n, c->io_a, c->partials, &grid);
   c->launches += launch_reduce_partials(c->stream, c->partials, grid, c->d_scalars);
   double ss;
   int rc = amgb_fetch_scalar(c, &ss);
   if (rc) return rc;
   *out = sqrt(ss);
   return AMGB_OK;
}

static bool has_additive_cycle(const amgb_ctx *c)
{
   const int s = c->opt.solver;
   return s == AMGB_SOLVER_MULTADD || s == AMGB_SOLVER_AFACX || s == AMGB_SOLVER_BPX || s == AMGB_SOLVER_ASYNC_MULTADD || s == AMGB_SOLVER_ASYNC_AFACX;
}

int amgb_cycle(amgb_ctx *c, const double *r_host, double *c_host)
{
   NEED_READY(c);
   if (!r_host || !c_host) return amgb_fail(c, AMGB_EINVAL, "null vector");
   if (!has_additive_cycle(c)) return amgb_fail(c, AMGB_EINVAL, "amgb_cycle applies the additive cycles (Multadd, AFACx, BPX); this context was set up for solver %d", c->opt.solver);
   const int n0 = c->A[0].nrows;
   CUDA_OK(c, cudaMemcpyAsync(c->r[0], r_host, sizeof(double) * n0, cudaMemcpyHostToDevice, c->stream));
   enq_cycle(c, c->cvec, false);
   CUDA_OK(c, cudaMemcpyAsync(c_host, c->cvec, sizeof(double) * n0, cudaMemcpyDeviceToHost, c->stream));
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   CUDA_OK(c, cudaGetLastError());
   return AMGB_OK;
}

// ---- asynchronous additive solve ACROSS GPUs (DMEM async Multadd, src/DMEM_Add.cpp:101-130,391-458) ----------
// The reference assigns MPI ranks to grids: every grid's rank group holds the hierarchy down to its level and
// full-length fine vectors, runs its own restrict -> smooth -> prolong chain on its private residual, and sends
// the fine-level correction to the other grids, which accumulate it whenever it arrives.  Here a GPU plays a
// grid's rank group: amgb_async_dist_correct(level) is one pass of AddCycle + DMEM_AddCorrect_LocalRes +
// DMEM_AddResidual_LocalRes for that level -- private copy of u, r = f - A_0 u, chain, and the correction is
// added into this GPU's u and into every peer's u with fp64 reductions over NVLink (k_push_correction).
// Nothing ever waits for a peer.
int amgb_ipc_export_solution(amgb_ctx *c, unsigned char handle64[64])
{
   NEED_READY(c);
   static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t size");
   cudaIpcMemHandle_t h;
   CUDA_OK(c, cudaIpcGetMemHandle(&h, c->u));
   memcpy(handle64, &h, 64);
   return AMGB_OK;
}

int amgb_ipc_open_peers(amgb_ctx *c, int npeers, const unsigned char *handles)
{
   NEED_READY(c);
   if (npeers < 0 || npeers > AMGB_MAX_PEERS || (npeers > 0 && !handles)) return amgb_fail(c, AMGB_EINVAL, "bad peer list");
   for (int p = 0; p < npeers; p++) {
      cudaIpcMemHandle_t h;
      memcpy(&h, handles + 64 * (size_t)p, 64);
      void *ptr = nullptr;
      CUDA_OK(c, cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
      c->peer_u.push_back((double *)ptr);
   }
   return AMGB_OK;
}

int amgb_async_dist_correct(amgb_ctx *c, int level)
{
   NEED_READY(c);
   const int L = c->L, n0 = c->A[0].nrows;
   if (level < 0 || level >= L) return amgb_fail(c, AMGB_EINVAL, "bad level");
   const amgb_options &o = c->opt;
   if (o.solver != AMGB_SOLVER_MULTADD || (o.smoother != AMGB_SMOOTH_JACOBI && o.smoother != AMGB_SMOOTH_L1_JACOBI))
      return amgb_fail(c, AMGB_EINVAL, "the cross-GPU asynchronous solve runs Multadd with (L1-)Jacobi smoothing");
   if (o.factor_restriction) return amgb_fail(c, AMGB_EINVAL, "the cross-GPU asynchronous solve reads the explicit Rbar_l (factor_restriction = 0)");
   if (level == L - 1 && L > 1) return AMGB_OK;           // SMEM convention: the coarsest level contributes nothing
   double *ul = c->u_outer;                                // private copy of the solution (level_vector[k].u)
   CUDA_OK(c, cudaMemcpyAsync(ul, c->u, sizeof(double) * n0, cudaMemcpyDeviceToDevice, c->stream));
   enq_spmv(c, c->A[0], false, ul, c->r[0], epi(-1.0, 1.0, c->f), false);
   for (int l = 0; l < level; l++) enq_spmv(c, c->R[l], false, c->r[l], c->r[l + 1], epi(1.0, 0.0, nullptr), false);
   enq_smooth_zero(c, level, c->r[level], c->e[level], o.num_fine_smooth_sweeps, c->symmetric, false, c->t[level], c->w[level]);
   for (int l = level - 1; l >= 0; l--) enq_spmv(c, c->P[l], false, c->e[l + 1], c->e[l], epi(1.0, 0.0, nullptr), false);
   PeerPtrs pp;
   pp.n = (int)c->peer_u.size();
   for (int p = 0; p < pp.n; p++) pp.p[p] = c->peer_u[p];
   c->launches += launch_push_correction(c->cfg, c->stream, n0, c->e[0], c->u, pp);
   CUDA_OK(c, cudaGetLastError());
   return AMGB_OK;
}

// ||f - A_0 u||_2 of the resident vectors (waits for everything enqueued on the context's stream)
int amgb_residual_norm(amgb_ctx *c, double *norm)
{
   NEED_READY(c);
   if (!norm) return amgb_fail(c, AMGB_EINVAL, "null output");
   enq_residual(c);
   double ss;
   int rc = amgb_fetch_scalar(c, &ss);
   if (rc) return rc;
   *norm = sqrt(ss);
   return AMGB_OK;
}

int amgb_stream_synchronize(amgb_ctx *c)
{
   NEED_READY(c);
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   return AMGB_OK;
}

// ---- EigsPower (src/SMEM_Cheby.cpp:410-518) --------------------------------------------------------
// Extreme eigenvalues of B*A by power iteration on the device, B = one application of the selected cycle
// from a zero guess.  Start vector all ones, `iters` normalise / apply steps, eig_max = <v, BAv>; a second
// pass deflated with u <- BAv - eig_max*v gives eig_min.  ChebySetup's mu = (beta+alpha)/(beta-alpha),
// delta = 2/(beta+alpha) (:48-49) are left to the caller.  Scratch: u_outer, y_outer, cvec.
int amgb_eigs_power(amgb_ctx *c, int iters, double *eig_min, double *eig_max)
{
   NEED_READY(c);
   if (iters < 1 || !eig_min || !eig_max) return amgb_fail(c, AMGB_EINVAL, "bad arguments");
   if (!has_additive_cycle(c)) return amgb_fail(c, AMGB_EINVAL, "amgb_eigs_power applies the additive cycles (Multadd, AFACx, BPX); this context was set up for solver %d", c->opt.solver);
   const int n0 = c->A[0].nrows;
   double *u = c->u_outer, *e = c->y_outer;
   double lam[2] = {0.0, 0.0};
   int rc, grid;
   for (int pass = 0; pass < 2; pass++) {
      std::vector<double> ones((size_t)n0, 1.0);
      CUDA_OK(c, cudaMemcpyAsync(u, ones.data(), sizeof(double) * n0, cudaMemcpyHostToDevice, c->stream));
      CUDA_OK(c, cudaStreamSynchronize(c->stream));
      for (int it = 1;; it++) {
         double ss;
         c->launches += launch_sumsq(c->cfg, c->stream, n0, u, c->partials, &grid);
         c->launches += launch_reduce_partials(c->stream, c->partials, grid, c->d_scalars);
         if ((rc = amgb_fetch_scalar(c, &ss))) return rc;
         c->launches += launch_axpby(c->cfg, c->stream, n0, 1.0 / sqrt(ss), u, 0.0, u, e);        // u /= |u|; e = u
         enq_spmv(c, c->A[0], false, u, c->r[0], epi(1.0, 0.0, nullptr), false);                   // f = A u
         enq_cycle(c, u, false);                                                                   // u = B f
         if (it == iters) break;
         if (pass == 1) c->launches += launch_axpby(c->cfg, c->stream, n0, -lam[0], e, 1.0, u, nullptr);
      }
      c->launches += launch_dot(c->cfg, c->stream, n0, e, u, c->partials, &grid);
      c->launches += launch_reduce_partials(c->stream, c->partials, grid, c->d_scalars);
      if ((rc = amgb_fetch_scalar(c, &lam[pass]))) return rc;
   }
   *eig_max = lam[0];
   *eig_min = lam[1];
   CUDA_OK(c, cudaGetLastError());
   return AMGB_OK;
}

// ---- SMEM_Solve, synchronous branch ----------------------------------------------------------------
int amgb_solve_sync(amgb_ctx *c, double tol, int max_cycles, int cheby_flag, double mu, double delta,
                    double *hist, int *n_cycles, double *solve_seconds)
{
   NEED_READY(c);
   if (max_cycles < 0) return amgb_fail(c, AMGB_EINVAL, "max_cycles < 0");
   const int n0 = c->A[0].nrows;
   int rc;
   if (c->opt.solver == AMGB_SOLVER_MULT) {
      if (cheby_flag) return amgb_fail(c, AMGB_EINVAL, "Chebyshev acceleration is wired for the additive cycles");
      if (c->opt.smoother == AMGB_SMOOTH_HYBRID_JGS) return amgb_fail(c, AMGB_EINVAL, "MULT runs with (L1-)Jacobi smoothing");
      CUDA_OK(c, cudaMemsetAsync(c->e[c->L - 1], 0, sizeof(double) * c->A[c->L - 1].nrows, c->stream));   // InitVectors
   }
   // r0 (src/SMEM_Solve.cpp:60-70)
   enq_residual(c);
   double ss;
   if ((rc = amgb_fetch_scalar(c, &ss))) return rc;
   const double r0 = sqrt(ss);
   if (hist) hist[0] = 1.0;
   int done = 0;
   double omega = 2.0;
   const double mu24 = 4.0 * mu * mu;
   if (cheby_flag) {
      CUDA_OK(c, cudaMemsetAsync(c->u_outer, 0, sizeof(double) * n0, c->stream));
      CUDA_OK(c, cudaMemsetAsync(c->y_outer, 0, sizeof(double) * n0, c->stream));
   }
   // one iteration = cycle + residual + norm; captured once, replayed as a graph
   cudaGraphExec_t gexec = nullptr;
   long long graph_nodes = 0;
   if (!cheby_flag) {
      if (!c->graph_exec) {
         cudaGraph_t g;
         long long before = c->launches;
         CUDA_OK(c, cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
         if (c->opt.solver == AMGB_SOLVER_MULT) enq_vcycle(c);
         else enq_cycle(c, c->u, true);
         enq_residual(c);
         cudaMemcpyAsync(c->h_scalars, c->d_scalars, sizeof(double), cudaMemcpyDeviceToHost, c->stream);
         CUDA_OK(c, cudaStreamEndCapture(c->stream, &g));
         c->graph_kernels = c->launches - before;
         c->launches = before;
         CUDA_OK(c, cudaGraphInstantiate(&c->graph_exec, g, 0));
         cudaGraphDestroy(g);
      }
      gexec = c->graph_exec;
      graph_nodes = c->graph_kernels;
   }
   CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
   for (int k = 1; k <= max_cycles; k++) {
      if (gexec) {
         CUDA_OK(c, cudaGraphLaunch(gexec, c->stream));
         c->launches += graph_nodes;
         CUDA_OK(c, cudaStreamSynchronize(c->stream));
         ss = c->h_scalars[0];
      } else {
         // Chebyshev acceleration (src/SMEM_Solve.cpp:169-188): cycle from a zero guess on the
         // current residual, then the three-term recurrence
         enq_cycle(c, c->cvec, false);
         c->launches += launch_cheby(c->cfg, c->stream, n0, omega, delta, c->cvec, c->u_outer, c->y_outer, c->u);
         omega = 1.0 / (1.0 - omega / mu24);
         enq_residual(c);
         if ((rc = amgb_fetch_scalar(c, &ss))) return rc;
      }
      done = k;
      const double rel = sqrt(ss) / r0;
      if (hist) hist[k] = rel;
      if (rel < tol) break;
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
}

int amgb_smem_solve(amgb_ctx *c, const double *f_host, double *u_host, double tol, int num_cycles,
                    double *hist, int *n_cycles, int *corrections, double *final_relres, double *solve_seconds)
{
   NEED_READY(c);
   if (!f_host || !u_host) return amgb_fail(c, AMGB_EINVAL, "null host buffers");
   const int n0 = c->A[0].nrows;
   int rc;
   CUDA_OK(c, cudaMemcpyAsync(c->f, f_host, sizeof(double) * n0, cudaMemcpyHostToDevice, c->stream));
   CUDA_OK(c, cudaMemsetAsync(c->u, 0, sizeof(double) * n0, c->stream));   // InitSolve: x0 = 0
   const int solver = c->opt.solver;
   int done = 0;
   double rel = 0.0;
   if (solver == AMGB_SOLVER_ASYNC_MULTADD || solver == AMGB_SOLVER_ASYNC_AFACX) {
      if ((rc = amgb_solve_async(c, num_cycles, AMGB_CONVERGE_LOCAL, corrections, &rel, solve_seconds))) return rc;
      done = num_cycles;
      // no per-iteration history exists for a chaotic iteration: the two ends only
      if (hist) { for (int k = 0; k <= num_cycles; k++) hist[k] = 0.0; hist[0] = 1.0; hist[num_cycles] = rel; }
   } else {
      std::vector<double> h((size_t)num_cycles + 1, 0.0);
      if ((rc = amgb_solve_sync(c, tol, num_cycles, 0, 1.0, 1.0, h.data(), &done, solve_seconds))) return rc;
      if (hist) memcpy(hist, h.data(), sizeof(double) * ((size_t)done + 1));
      if (corrections) for (int l = 0; l < c->L; l++) corrections[l] = done;   // src/SMEM_Solve.cpp:246-248
      rel = h[done];
   }
   if (n_cycles) *n_cycles = done;
   if (final_relres) *final_relres = rel;
   CUDA_OK(c, cudaMemcpyAsync(u_host, c->u, sizeof(double) * n0, cudaMemcpyDeviceToHost, c->stream));
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   return AMGB_OK;
}

int amgb_time_residual(amgb_ctx *c, int reps, double *ms_per_launch)
{
   NEED_READY(c);
   if (reps < 1 || !ms_per_launch) return amgb_fail(c, AMGB_EINVAL, "bad arguments");
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
   for (int k = 0; k < reps; k++) {
      int grid;
      c->launches += launch_spmv(c->cfg, c->stream, c->A[0], false, c->u, c->r[0], epi(-1.0, 1.0, c->f), c->partials, &grid);
   }
   CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
   CUDA_OK(c, cudaEventSynchronize(c->ev1));
   float ms = 0;
   cudaEventElapsedTime(&ms, c->ev0, c->ev1);
   *ms_per_launch = ms / reps;
   return AMGB_OK;
}

// event-timed y = M x (plain epilogue) for one matrix of the hierarchy: the tuning harness's probe
int amgb_time_spmv(amgb_ctx *c, int kind, int level, int use_sval, int reps, double *ms_per_launch)
{
   NEED_READY(c);
   if (level < 0 || level >= c->L || (kind != AMGB_MAT_A && level >= c->L - 1) || reps < 1 || !ms_per_launch)
      return amgb_fail(c, AMGB_EINVAL, "bad arguments");
   const DevCSR &M = kind == AMGB_MAT_A ? c->A[level] : (kind == AMGB_MAT_P ? c->P[level] : c->R[level]);
   if (use_sval < 0 || use_sval > 4 || (use_sval > 1 && use_sval < 4 && kind != AMGB_MAT_A) || (use_sval == 4 && kind != AMGB_MAT_P))
      return amgb_fail(c, AMGB_EINVAL, "bad arguments");
   const bool sval = use_sval >= 1 && use_sval <= 3;
   if (sval && !M.sval && !M.sell_sval) return amgb_fail(c, AMGB_EINVAL, "no scaled values for this matrix");
   const double *x = kind == AMGB_MAT_A ? c->r[level] : (kind == AMGB_MAT_P ? c->e[level + 1] : c->r[level]);
   double *y = kind == AMGB_MAT_A ? c->e[level] : (kind == AMGB_MAT_P ? c->t[level] : c->t[level + 1]);
   const double *rs = (c->opt.smoother == AMGB_SMOOTH_L1_JACOBI) ? c->inv_l1[level] : c->ws[level];
   // 2: the symmetrised smoother's pass as the explicit cycle launches it; 3: the factorised restriction's pass (t and e);
   // 4: the Horner prolongation's e_l += P_l e_{l+1} (in place, as enq_cycle launches it)
   const SpmvEpilogue e = use_sval == 2 ? epi(-1.0, 2.0, x, 0.0, nullptr, rs)
                          : (use_sval == 3 ? epi(-1.0, 1.0, x) : (use_sval == 4 ? epi(1.0, 1.0, c->e[level]) : epi(1.0, 0.0, nullptr)));
   double *y1 = use_sval == 3 ? c->t[level] : (use_sval == 4 ? c->e[level] : y), *y2 = use_sval == 3 ? c->e[level] : nullptr;
   int grid;
   for (int k = 0; k < 3; k++) c->launches += launch_spmv(c->cfg, c->stream, M, sval, x, y1, e, nullptr, &grid, nullptr, y2, rs);
   CUDA_OK(c, cudaStreamSynchronize(c->stream));
   CUDA_OK(c, cudaEventRecord(c->ev0, c->stream));
   for (int k = 0; k < reps; k++) c->launches += launch_spmv(c->cfg, c->stream, M, sval, x, y1, e, nullptr, &grid, nullptr, y2, rs);
   CUDA_OK(c, cudaEventRecord(c->ev1, c->stream));
   CUDA_OK(c, cudaEventSynchronize(c->ev1));
   float ms = 0;
   cudaEventElapsedTime(&ms, c->ev0, c->ev1);
   *ms_per_launch = ms / reps;
   CUDA_OK(c, cudaGetLastError());
   return AMGB_OK;
}

// one product with every epilogue operand launch_spmv takes, host in / host out (tests of the SpMV paths)
int amgb_spmv_probe(amgb_ctx *c, int kind, int level, int use_sval, const double *coef, const double *x, const double *b,
                    const double *cc, const double *rs, const double *b2, const double *xs, const double *w, int mode, double *y,
                    double *y2, double *sum, int *window_path)
{
   NEED_READY(c);
   if (level < 0 || level >= c->L || (kind != AMGB_MAT_A && level >= c->L - 1)) return amgb_fail(c, AMGB_EINVAL, "bad level");
   const DevCSR &M = kind == AMGB_MAT_A ? c->A[level] : (kind == AMGB_MAT_P ? c->P[level] : c->R[level]);
   if (!coef || !x || !y || mode < 0 || mode > 3 || (mode >= 2 && !w) || ((mode == 1 || mode == 2) && !sum) ||
       (mode == 3 && (!b || !y2 || !use_sval)))
      return amgb_fail(c, AMGB_EINVAL, "bad probe arguments");
   if (use_sval && !M.sval && !M.sell_sval) return amgb_fail(c, AMGB_EINVAL, "no scaled values for this matrix");
   const size_t nr = M.nrows, nc = M.ncols;
   const double *host[8] = {x, b, cc, rs, b2, xs, mode == 1 ? nullptr : w, nullptr};
   const size_t len[8] = {nc, nr, nr, nr, nr, nr, nr, nr};
   double *dev[8] = {};
   int rc = AMGB_OK;
   double *dy = nullptr, *dy2 = nullptr;
   for (int i = 0; i < 7 && rc == AMGB_OK; i++)
      if (host[i]) {
         if (cudaMalloc((void **)&dev[i], sizeof(double) * len[i]) != cudaSuccess) rc = AMGB_ECUDA;
         else if (cudaMemcpyAsync(dev[i], host[i], sizeof(double) * len[i], cudaMemcpyHostToDevice, c->stream) != cudaSuccess) rc = AMGB_ECUDA;
      }
   if (rc == AMGB_OK && cudaMalloc((void **)&dy, sizeof(double) * nr) != cudaSuccess) rc = AMGB_ECUDA;
   if (rc == AMGB_OK && mode == 3 && cudaMalloc((void **)&dy2, sizeof(double) * nr) != cudaSuccess) rc = AMGB_ECUDA;
   if (rc == AMGB_OK) {
      SpmvEpilogue e = epi(coef[0], coef[1], dev[1], coef[2], dev[2], dev[3]);
      e.beta2 = coef[3]; e.b2 = dev[4];
      e.xself = coef[4]; e.xs = dev[5];
      int grid = 0;
      if (window_path) *window_path = spmv_window_path(c->cfg, M) ? 1 : 0;
      c->launches += launch_spmv(c->cfg, c->stream, M, use_sval != 0, dev[0], dy, e, mode == 1 || mode == 2 ? c->partials : nullptr,
                                 &grid, mode == 2 ? dev[6] : nullptr, dy2, mode == 3 ? dev[6] : nullptr);
      if (mode == 1 || mode == 2) c->launches += launch_reduce_partials(c->stream, c->partials, grid, c->d_scalars);
      if (cudaMemcpyAsync(y, dy, sizeof(double) * nr, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess) rc = AMGB_ECUDA;
      if (rc == AMGB_OK && dy2 && cudaMemcpyAsync(y2, dy2, sizeof(double) * nr, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess) rc = AMGB_ECUDA;
      if (rc == AMGB_OK && (mode == 1 || mode == 2)) rc = amgb_fetch_scalar(c, sum);
      if (rc == AMGB_OK && cudaStreamSynchronize(c->stream) != cudaSuccess) rc = AMGB_ECUDA;
   }
   cudaStreamSynchronize(c->stream);
   for (double *p : dev) cudaFree(p);
   cudaFree(dy);
   cudaFree(dy2);
   if (rc == AMGB_ECUDA) return amgb_fail(c, rc, "spmv probe: %s", cudaGetErrorString(cudaGetLastError()));
   return rc;
}

// bytes of coarse-hierarchy data placed in the L2-pinned arena (the access-policy window of the persistent kernel)
int amgb_l2_arena_bytes(amgb_ctx *c, long long *used, long long *capacity)
{
   if (!c) return AMGB_EINVAL;
   if (used) *used = (long long)c->arena_used;
   if (capacity) *capacity = (long long)c->arena_size;
   return AMGB_OK;
}

// slices stored in the SELL-U encoding and their groups, over the whole hierarchy
int amgb_sellu_stats(amgb_ctx *c, long long *slices, long long *groups)
{
   if (!c) return AMGB_EINVAL;
   if (slices) *slices = c->sellu_slices;
   if (groups) *groups = c->sellu_groups;
   return AMGB_OK;
}

int amgb_level_storage(amgb_ctx *c, int kind, int level, int *is_sell)
{
   if (!c || level < 0 || level >= c->L || !is_sell) return AMGB_EINVAL;
   const DevCSR &M = kind == AMGB_MAT_A ? c->A[level] : (kind == AMGB_MAT_P ? c->P[level] : c->R[level]);
   *is_sell = M.sell_slices > 0;
   return AMGB_OK;
}

}  // extern "C"
